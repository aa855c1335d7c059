"""ctypes view of the C ABI in include/ookd_gpu.h (libookd_gpu.so).

This module is glue for tests, bench.py and scripting; the product is the
shared library.  It contains no arithmetic of its own and no fallback: if the
library is missing it is built, and if there is no sm_100 device every compute
call raises OokdError.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OOKD_GPU_LIB") or os.path.join(_HERE, "lib", "libookd_gpu.so")

MAX_STAGES = 8
MSG_BYTES = 32
K_INF = 0xFFFFFFFF
LEVEL_BINS = 4096
LEVEL_MARGIN_DB = 12.0
DEGLITCH_MAX = 65535

FLAG_FORCE_GENERIC = 1
FLAG_NO_SCREEN = 2
FLAG_NO_TMA = 8
FLAG_SYNC_TAIL = 16
FLAG_SHARE_SMS = 32
FLAG_NO_GRAPH = 64
FLAG_FUSED_SM = 128
FLAG_FMA_SCREEN = 256
FLAG_NO_ADAPTIVE = 512
FLAG_INPUT_CS8 = 1024
FLAG_INPUT_CU8 = 2048

# input_format -> (ookd_gpu_config.flags bit, numpy dtype of a host capture); every format is interleaved I,Q
INPUT_FORMATS = {"sc16q11": (0, np.int16), "cs8": (FLAG_INPUT_CS8, np.int8), "cu8": (FLAG_INPUT_CU8, np.uint8)}

# every symbol include/ookd_gpu.h declares
EXPORTS = [
    "ookd_sm_compile", "ookd_sm_compiled_free", "ookd_sm_idle_carry", "ookd_power_threshold",
    "ookd_tune_step", "ookd_tune_sc16q11", "ookd_level_threshold", "ookd_gpu_levels",
    "ookd_gpu_device_count", "ookd_gpu_strerror", "ookd_gpu_last_error",
    "ookd_gpu_create", "ookd_gpu_destroy", "ookd_gpu_decode", "ookd_gpu_decode_shard",
    "ookd_gpu_decode_begin", "ookd_gpu_decode_end", "ookd_gpu_batch_decode",
    "ookd_gpu_resolve", "ookd_gpu_halo", "ookd_gpu_input_bytes", "ookd_gpu_total_decimation", "ookd_gpu_initial_carry",
    "ookd_gpu_edges", "ookd_gpu_bits", "ookd_gpu_filtered", "ookd_gpu_filter_cf", "ookd_gpu_synth", "ookd_gpu_synth_ex",
    "ookd_gpu_host_alloc", "ookd_gpu_host_free", "ookd_gpu_dev_alloc", "ookd_gpu_dev_free",
    "ookd_gpu_memcpy_h2d", "ookd_gpu_memcpy_d2h", "ookd_gpu_filtered_sc16q11",
    "ookd_gpu_multi_create", "ookd_gpu_multi_destroy", "ookd_gpu_multi_halo", "ookd_gpu_multi_n_gpus",
    "ookd_gpu_multi_handle", "ookd_gpu_multi_shards_used", "ookd_gpu_multi_last_error", "ookd_gpu_multi_shard_range",
    "ookd_gpu_multi_decode", "ookd_gpu_multi_edges",
    "ookd_gpu_multi_decode_begin", "ookd_gpu_multi_decode_end", "ookd_gpu_multi_resolve",
]


class OokdError(RuntimeError):
    pass


class FilterDesc(C.Structure):
    _fields_ = [("num_stages", C.c_uint32),
                ("decimation", C.c_uint32 * MAX_STAGES),
                ("num_taps", C.c_uint32 * MAX_STAGES),
                ("taps", C.POINTER(C.c_float) * MAX_STAGES)]


class SmTriggerUs(C.Structure):
    _fields_ = [("cond", C.c_int32), ("action", C.c_int32), ("next_state", C.c_uint32),
                ("reserved", C.c_uint32), ("duration_us", C.c_uint64)]


class SmStateUs(C.Structure):
    _fields_ = [("duration_us", C.c_uint64), ("timeout_us", C.c_uint64),
                ("first_trigger", C.c_uint32), ("num_triggers", C.c_uint32)]


class SmDesc(C.Structure):
    _fields_ = [("num_states", C.c_uint32), ("num_triggers", C.c_uint32),
                ("states", C.POINTER(SmStateUs)), ("triggers", C.POINTER(SmTriggerUs)),
                ("max_bits", C.c_uint32), ("sample_rate", C.c_uint32)]


class SmTriggerK(C.Structure):
    _fields_ = [("cond", C.c_int32), ("action", C.c_int32), ("next_state", C.c_uint32),
                ("kmin", C.c_uint32), ("kmax", C.c_uint32)]


class SmStateK(C.Structure):
    _fields_ = [("first_trigger", C.c_uint32), ("num_triggers", C.c_uint32),
                ("dmin", C.c_uint32), ("dmax", C.c_uint32), ("ktimeout", C.c_uint32), ("ksat", C.c_uint32)]


class SmCompiled(C.Structure):
    _fields_ = [("num_states", C.c_uint32), ("num_triggers", C.c_uint32),
                ("states", C.POINTER(SmStateK)), ("triggers", C.POINTER(SmTriggerK)),
                ("max_bits", C.c_uint32), ("k_sat", C.c_uint32)]


class Msg(C.Structure):
    _fields_ = [("out_sample", C.c_uint64), ("buffer_idx", C.c_uint64), ("num_bits", C.c_uint32),
                ("reserved", C.c_uint32), ("data", C.c_uint8 * MSG_BYTES)]


MSG_DTYPE = np.dtype([("out_sample", "<u8"), ("buffer_idx", "<u8"), ("num_bits", "<u4"), ("reserved", "<u4"),
                      ("data", "u1", (MSG_BYTES,))])
assert MSG_DTYPE.itemsize == C.sizeof(Msg)


def msgs_to_tuples(rec, nbytes):
    """Structured message array -> [(out_sample, buffer_idx, num_bits, data bytes)]."""
    return list(zip(rec["out_sample"].tolist(), rec["buffer_idx"].tolist(), rec["num_bits"].tolist(),
                    [bytes(d[:nbytes]) for d in rec["data"]]))


class SmCarry(C.Structure):
    _fields_ = [("state", C.c_uint32), ("k", C.c_uint32), ("num_bits", C.c_uint32),
                ("prev_bit", C.c_uint32), ("data", C.c_uint8 * MSG_BYTES)]

    def astuple(self):
        return (self.state, self.k, self.num_bits, self.prev_bit, bytes(self.data))

    @classmethod
    def fromtuple(cls, t):
        c = cls()
        c.state, c.k, c.num_bits, c.prev_bit = t[:4]
        C.memmove(c.data, t[4], MSG_BYTES)
        return c


class GpuConfig(C.Structure):
    """struct ookd_gpu_config up to tune_step, the layout of earlier releases.  The whole struct is GpuConfigEx below:
    use it for new code (Gpu and MultiGpu do)."""
    _fields_ = [("filter", C.POINTER(FilterDesc)), ("sm", C.POINTER(SmDesc)), ("threshold", C.c_float),
                ("samples_per_buffer", C.c_uint32), ("device_id", C.c_int32), ("flags", C.c_uint32),
                ("sm_chunk_buffers", C.c_uint32), ("sm_warmup", C.c_uint32), ("sm_burst_rounds", C.c_uint32),
                ("sub_windows", C.c_uint32), ("tune_step", C.c_uint32)]


class GpuConfigEx(C.Structure):
    """struct ookd_gpu_config with every field.  GpuConfig ends at tune_step: the appended deglitch lies in its tail
    padding (both are 56 bytes), which ctypes zero-fills, so a GpuConfig still describes a handle with deglitch = 0."""
    _fields_ = GpuConfig._fields_ + [("deglitch", C.c_uint32)]


assert C.sizeof(GpuConfigEx) == C.sizeof(GpuConfig)


class GpuResult(C.Structure):
    _fields_ = [("n_in", C.c_uint64), ("n_out", C.c_uint64), ("n_buffers", C.c_uint64),
                ("n_edges", C.c_uint64), ("n_msgs", C.c_uint64), ("msgs", C.POINTER(Msg)),
                ("first_bit", C.c_uint32), ("sm_rounds", C.c_uint32), ("kernel_ms", C.c_float),
                ("fir_ms", C.c_float), ("gpu_launches", C.c_uint32), ("refined_tiles", C.c_uint32),
                ("refined_blocks", C.c_uint32), ("entry_is_provisional", C.c_uint32), ("entry_used", SmCarry),
                ("screen_ms", C.c_float), ("host_syncs", C.c_uint32), ("fir_mode", C.c_uint32)]


class Capture(C.Structure):
    _fields_ = [("iq", C.c_void_p), ("n_samples", C.c_uint64), ("iq_is_device_ptr", C.c_int32), ("handle", C.c_uint32)]


def build_library():
    subprocess.run(["make", "-s", "-C", os.path.join(_HERE, "csrc")], check=True)


_lib = None


def lib():
    """Load libookd_gpu.so (building it first if absent).  Never falls back to anything else."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build_library()
        L = C.CDLL(LIB_PATH)
        L.ookd_sm_compile.restype = C.c_int
        L.ookd_sm_compile.argtypes = [C.POINTER(SmDesc), C.POINTER(SmCompiled)]
        L.ookd_sm_compiled_free.argtypes = [C.POINTER(SmCompiled)]
        L.ookd_sm_idle_carry.argtypes = [C.POINTER(SmCompiled), C.POINTER(SmCarry)]
        L.ookd_power_threshold.restype = C.c_float
        L.ookd_power_threshold.argtypes = [C.c_float]
        L.ookd_tune_step.restype = C.c_int
        L.ookd_tune_step.argtypes = [C.c_double, C.c_uint32, C.POINTER(C.c_uint32)]
        L.ookd_tune_sc16q11.restype = C.c_int
        L.ookd_tune_sc16q11.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32]
        L.ookd_level_threshold.restype = C.c_int
        L.ookd_level_threshold.argtypes = [C.c_void_p, C.c_double, C.POINTER(C.c_float), C.POINTER(C.c_double)]
        L.ookd_gpu_levels.restype = C.c_int
        L.ookd_gpu_levels.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_void_p]
        L.ookd_gpu_device_count.restype = C.c_int
        L.ookd_gpu_strerror.restype = C.c_char_p
        L.ookd_gpu_strerror.argtypes = [C.c_int]
        L.ookd_gpu_last_error.restype = C.c_char_p
        L.ookd_gpu_last_error.argtypes = [C.c_void_p]
        L.ookd_gpu_create.restype = C.c_int
        L.ookd_gpu_create.argtypes = [C.POINTER(C.c_void_p), C.c_void_p]              # GpuConfig or GpuConfigEx
        L.ookd_gpu_destroy.argtypes = [C.c_void_p]
        L.ookd_gpu_decode.restype = C.c_int
        L.ookd_gpu_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.POINTER(GpuResult)]
        L.ookd_gpu_decode_shard.restype = C.c_int
        L.ookd_gpu_decode_shard.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int,
                                            C.POINTER(SmCarry), C.POINTER(SmCarry), C.POINTER(GpuResult)]
        L.ookd_gpu_decode_begin.restype = C.c_int
        L.ookd_gpu_decode_begin.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int,
                                            C.POINTER(SmCarry)]
        L.ookd_gpu_decode_end.restype = C.c_int
        L.ookd_gpu_decode_end.argtypes = [C.c_void_p, C.POINTER(SmCarry), C.POINTER(GpuResult)]
        L.ookd_gpu_batch_decode.restype = C.c_int
        L.ookd_gpu_batch_decode.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(Capture), C.c_uint32,
                                            C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(GpuResult)]
        L.ookd_gpu_resolve.restype = C.c_int
        L.ookd_gpu_resolve.argtypes = [C.c_void_p, C.POINTER(SmCarry), C.POINTER(SmCarry), C.POINTER(GpuResult)]
        L.ookd_gpu_halo.restype = C.c_uint32
        L.ookd_gpu_halo.argtypes = [C.c_void_p]
        L.ookd_gpu_total_decimation.restype = C.c_uint32
        L.ookd_gpu_input_bytes.argtypes = [C.c_void_p]
        L.ookd_gpu_input_bytes.restype = C.c_uint32
        L.ookd_gpu_total_decimation.argtypes = [C.c_void_p]
        L.ookd_gpu_initial_carry.argtypes = [C.c_void_p, C.POINTER(SmCarry)]
        L.ookd_gpu_edges.restype = C.c_int
        L.ookd_gpu_edges.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_uint64)), C.POINTER(C.c_uint64),
                                     C.POINTER(C.c_uint32)]
        L.ookd_gpu_bits.restype = C.c_int
        L.ookd_gpu_bits.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.ookd_gpu_filtered.restype = C.c_int
        L.ookd_gpu_filtered.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                        C.POINTER(C.c_uint64)]
        L.ookd_gpu_filter_cf.restype = C.c_int
        L.ookd_gpu_filter_cf.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                         C.POINTER(C.c_uint64)]
        L.ookd_gpu_synth.restype = C.c_int
        L.ookd_gpu_synth.argtypes = [C.c_int32, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_void_p,
                                     C.c_uint64, C.c_int32, C.c_int32, C.c_int32, C.c_uint64]
        L.ookd_gpu_synth_ex.restype = C.c_int
        L.ookd_gpu_synth_ex.argtypes = [C.c_int32, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_void_p,
                                        C.c_uint64, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_uint32]
        L.ookd_gpu_filtered_sc16q11.restype = C.c_int
        L.ookd_gpu_filtered_sc16q11.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.ookd_gpu_multi_create.restype = C.c_int
        L.ookd_gpu_multi_create.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(C.c_int32), C.c_uint32]
        L.ookd_gpu_multi_destroy.argtypes = [C.c_void_p]
        L.ookd_gpu_multi_halo.restype = C.c_uint32
        L.ookd_gpu_multi_halo.argtypes = [C.c_void_p]
        L.ookd_gpu_multi_n_gpus.restype = C.c_uint32
        L.ookd_gpu_multi_n_gpus.argtypes = [C.c_void_p]
        L.ookd_gpu_multi_handle.restype = C.c_void_p
        L.ookd_gpu_multi_handle.argtypes = [C.c_void_p, C.c_uint32]
        L.ookd_gpu_multi_shards_used.restype = C.c_uint32
        L.ookd_gpu_multi_shards_used.argtypes = [C.c_void_p]
        L.ookd_gpu_multi_last_error.restype = C.c_char_p
        L.ookd_gpu_multi_last_error.argtypes = [C.c_void_p]
        L.ookd_gpu_multi_shard_range.restype = C.c_int
        L.ookd_gpu_multi_shard_range.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint64),
                                                 C.POINTER(C.c_uint64)]
        L.ookd_gpu_multi_decode.restype = C.c_int
        L.ookd_gpu_multi_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int,
                                            C.POINTER(SmCarry), C.POINTER(SmCarry), C.POINTER(GpuResult)]
        L.ookd_gpu_multi_edges.restype = C.c_int
        L.ookd_gpu_multi_edges.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_uint64)), C.POINTER(C.c_uint64),
                                           C.POINTER(C.c_uint32)]
        L.ookd_gpu_host_alloc.restype = C.c_void_p
        L.ookd_gpu_host_alloc.argtypes = [C.c_size_t]
        L.ookd_gpu_host_free.argtypes = [C.c_void_p]
        L.ookd_gpu_dev_alloc.restype = C.c_void_p
        L.ookd_gpu_dev_alloc.argtypes = [C.c_int32, C.c_size_t]
        L.ookd_gpu_dev_free.argtypes = [C.c_int32, C.c_void_p]
        L.ookd_gpu_memcpy_h2d.restype = C.c_int
        L.ookd_gpu_memcpy_h2d.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t]
        L.ookd_gpu_memcpy_d2h.restype = C.c_int
        L.ookd_gpu_memcpy_d2h.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t]
        _lib = L
    return _lib


def make_filter_desc(stages):
    """stages: [(decimation, float32 taps)] -> (FilterDesc, keepalive)."""
    fd = FilterDesc()
    keep = []
    fd.num_stages = len(stages)
    for i, (dec, taps) in enumerate(stages):
        t = np.ascontiguousarray(taps, dtype=np.float32)
        keep.append(t)
        fd.decimation[i] = int(dec)
        fd.num_taps[i] = len(t)
        fd.taps[i] = t.ctypes.data_as(C.POINTER(C.c_float))
    return fd, keep


def make_sm_desc(states, num_bits, sample_rate):
    """states: [dict(duration_us, timeout_us, triggers=[dict(cond, action, next, duration_us)])]
    (state 0 = RESET) -> (SmDesc, keepalive)."""
    nt = sum(len(s["triggers"]) for s in states)
    st = (SmStateUs * len(states))()
    tr = (SmTriggerUs * max(nt, 1))()
    q = 0
    for i, s in enumerate(states):
        st[i].duration_us = int(s["duration_us"])
        st[i].timeout_us = int(s["timeout_us"])
        st[i].first_trigger = q
        st[i].num_triggers = len(s["triggers"])
        for t in s["triggers"]:
            tr[q].cond = int(t["cond"])
            tr[q].action = int(t["action"])
            tr[q].next_state = int(t["next"])
            tr[q].duration_us = int(t["duration_us"])
            q += 1
    d = SmDesc()
    d.num_states = len(states)
    d.num_triggers = nt
    d.states = C.cast(st, C.POINTER(SmStateUs))
    d.triggers = C.cast(tr, C.POINTER(SmTriggerUs))
    d.max_bits = int(num_bits)
    d.sample_rate = int(sample_rate)
    return d, (st, tr)


def sm_compile(states, num_bits, sample_rate):
    """Host-only: integer windows the GPU will use.  -> dict(states=[...], triggers=[...], k_sat)."""
    d, keep = make_sm_desc(states, num_bits, sample_rate)
    out = SmCompiled()
    rc = lib().ookd_sm_compile(C.byref(d), C.byref(out))
    if rc != 0:
        raise OokdError(f"ookd_sm_compile: {lib().ookd_gpu_strerror(rc).decode()}")
    res = dict(k_sat=out.k_sat, max_bits=out.max_bits,
               states=[dict(first_trigger=out.states[i].first_trigger, num_triggers=out.states[i].num_triggers,
                            dmin=out.states[i].dmin, dmax=out.states[i].dmax, ktimeout=out.states[i].ktimeout,
                            ksat=out.states[i].ksat)
                       for i in range(out.num_states)],
               triggers=[dict(cond=out.triggers[i].cond, action=out.triggers[i].action,
                              next=out.triggers[i].next_state, kmin=out.triggers[i].kmin, kmax=out.triggers[i].kmax)
                         for i in range(out.num_triggers)])
    lib().ookd_sm_compiled_free(C.byref(out))
    return res


def sm_idle_carry(states, num_bits, sample_rate):
    """Host-only: the state the compiled machine settles in on a constant-0 input from RESET (the stitcher's
    speculative seed).  -> carry tuple (state, k, num_bits, prev_bit, data32)."""
    d, keep = make_sm_desc(states, num_bits, sample_rate)
    out = SmCompiled()
    rc = lib().ookd_sm_compile(C.byref(d), C.byref(out))
    if rc != 0:
        raise OokdError(f"ookd_sm_compile: {lib().ookd_gpu_strerror(rc).decode()}")
    c = SmCarry()
    lib().ookd_sm_idle_carry(C.byref(out), C.byref(c))
    lib().ookd_sm_compiled_free(C.byref(out))
    return c.astuple()


def power_threshold(thr):
    return float(lib().ookd_power_threshold(C.c_float(thr)))


def tune_step(offset_hz, samplerate):
    """Phase step of a transmitter offset_hz from the capture's centre at samplerate samples/s (ookd_tune_step):
    llround(offset_hz / samplerate * 2^32) modulo 2^32.  ValueError if offset_hz is not finite, samplerate is 0 or
    |offset_hz| >= samplerate / 2."""
    if not 0 <= int(samplerate) < 2**32:
        raise ValueError(f"samplerate {samplerate} is not a uint32")
    step = C.c_uint32()
    if lib().ookd_tune_step(C.c_double(float(offset_hz)), C.c_uint32(int(samplerate)), C.byref(step)) != 0:
        raise ValueError(f"no tune step for an offset of {offset_hz} Hz at {samplerate} samples/s: the offset must be "
                         f"finite and below half the sample rate in magnitude")
    return int(step.value)


def tune_sc16q11(iq, first_sample, step):
    """CPU form of the tuning rotation T (ookd_tune_sc16q11): int16 I,Q samples whose first one is global sample
    first_sample -> the rotated samples, same shape."""
    a = np.ascontiguousarray(iq, dtype=np.int16)
    out = np.empty_like(a)
    rc = lib().ookd_tune_sc16q11(C.c_void_p(a.ctypes.data), C.c_void_p(out.ctypes.data), C.c_uint64(int(first_sample)),
                                 C.c_uint64(a.size // 2), C.c_uint32(int(step)))
    if rc != 0:
        raise OokdError(f"ookd_tune_sc16q11: {lib().ookd_gpu_strerror(rc).decode()}")
    return out


def level_threshold(hist, margin_db=LEVEL_MARGIN_DB):
    """Threshold rule of include/ookd_gpu.h, "Levels": a level histogram (LEVEL_BINS counts) -> (threshold, floor_power),
    the float to create decode handles with and F, the upper edge of the median bin.  ValueError where
    ookd_level_threshold returns OOKD_ERR_ARG: no counts, a median in the inf / NaN bins, a non-finite margin or
    threshold, or more counts than a uint64 holds."""
    h = np.asarray(hist)
    if h.shape != (LEVEL_BINS,) or (h.dtype.kind not in "ui") or (h.dtype.kind == "i" and (h < 0).any()):
        raise ValueError(f"a level histogram is {LEVEL_BINS} non-negative integer counts")
    h = np.ascontiguousarray(h, dtype=np.uint64)
    thr, floor = C.c_float(), C.c_double()
    if lib().ookd_level_threshold(C.c_void_p(h.ctypes.data), C.c_double(float(margin_db)), C.byref(thr),
                                  C.byref(floor)) != 0:
        raise ValueError(f"no threshold from this histogram ({int(h.sum(dtype=np.float64))} outputs) at a margin of "
                         f"{margin_db} dB: it needs outputs, a finite median power, and a finite margin and result")
    return float(thr.value), float(floor.value)


def device_count():
    return int(lib().ookd_gpu_device_count())


def _input_format(input_format, flags=0):
    """input_format name -> (flag, numpy dtype).  The format is chosen by name only: format bits in `flags` would make
    the handle read bytes while this binding still passed int16 arrays."""
    if flags & (FLAG_INPUT_CS8 | FLAG_INPUT_CU8):
        raise ValueError("choose the capture format with input_format=, not with the OOKD_FLAG_INPUT_* bits in flags")
    if input_format not in INPUT_FORMATS:
        raise ValueError(f"input_format must be one of {sorted(INPUT_FORMATS)}, not {input_format!r}")
    return INPUT_FORMATS[input_format]


def _host_iq(iq, input_format="sc16q11"):
    """Host capture -> flat contiguous array of the format's dtype (I, Q interleaved; shape (n, 2) or flat).
    8-bit captures must already have their dtype (int8 for cs8, uint8 for cu8): converting values between formats is
    not a cast, so any other dtype -- and an 8-bit array handed to an SC16Q11 handle -- is a ValueError."""
    dtype = _input_format(input_format)[1]
    got = getattr(iq, "dtype", None)
    if input_format != "sc16q11" and got != dtype:
        raise ValueError(f"a {input_format} capture is a numpy {np.dtype(dtype).name} array, not {got}")
    if input_format == "sc16q11" and got in (np.dtype(np.int8), np.dtype(np.uint8)):
        raise ValueError(f"a {got} array is an 8-bit capture: decode it with a handle created with input_format="
                         f"{'cs8' if got == np.dtype(np.int8) else 'cu8'!r}")
    return np.ascontiguousarray(iq, dtype=dtype).reshape(-1)


def _as_ptr(iq, input_format="sc16q11"):
    """numpy capture -> (pointer, n_samples, is_device=0, keepalive); (int ptr, n) tuples pass through as device."""
    if isinstance(iq, tuple):
        return C.c_void_p(int(iq[0])), int(iq[1]), 1, None
    a = _host_iq(iq, input_format)
    return C.c_void_p(a.ctypes.data), a.size // 2, 0, a


class Gpu:
    """One ookd_gpu handle.  input_format: "sc16q11" (int16 I,Q), "cs8" (int8 I,Q) or "cu8" (uint8 I,Q) host arrays;
    an 8-bit capture decodes exactly as its widened SC16Q11 capture does (include/ookd_gpu.h, OOKD_FLAG_INPUT_*).
    tune_step != 0 (see tune_step()): decode the capture shifted down by that frequency offset, exactly as the untuned
    handle decodes the rotated capture T(x) (include/ookd_gpu.h, "Tuning").
    deglitch = M >= 1: every consumer of decisions sees the majority of the last 2M+1 (include/ookd_gpu.h,
    "Deglitch"); M > DEGLITCH_MAX is an OokdError from ookd_gpu_create."""

    def __init__(self, filter_stages=None, sm=None, threshold=0.1, samples_per_buffer=8192, device_id=-1,
                 flags=0, sm_chunk_buffers=0, sm_warmup=0, sm_burst_rounds=0, sub_windows=0, input_format="sc16q11",
                 tune_step=0, deglitch=0):
        flags |= _input_format(input_format, flags)[0]
        self.input_format = input_format
        L = lib()
        cfg = GpuConfigEx()
        self._keep = []
        if filter_stages:
            fd, k = make_filter_desc(filter_stages)
            self._keep += [fd, k]
            cfg.filter = C.pointer(fd)
        if sm is not None:
            sd, k = make_sm_desc(sm["states"], sm["num_bits"], sm["sample_rate"])
            self._keep += [sd, k]
            cfg.sm = C.pointer(sd)
            self.msg_bytes = (sm["num_bits"] + 7) // 8
        else:
            self.msg_bytes = 0
        cfg.threshold = threshold
        cfg.samples_per_buffer = samples_per_buffer
        cfg.device_id = device_id
        cfg.flags = flags
        cfg.sm_chunk_buffers = sm_chunk_buffers
        cfg.sm_warmup = sm_warmup
        cfg.sm_burst_rounds = sm_burst_rounds
        cfg.sub_windows = sub_windows
        cfg.tune_step = tune_step
        cfg.deglitch = deglitch
        self.h = C.c_void_p()
        rc = L.ookd_gpu_create(C.byref(self.h), C.byref(cfg))
        if rc != 0:
            self.h = None
            raise OokdError(f"ookd_gpu_create: {L.ookd_gpu_strerror(rc).decode()}")
        self.device_id = device_id
        self.want_list = True        # build res["msgs"] (list of tuples) besides res["msgs_raw"]

    def close(self):
        # (at interpreter shutdown module globals may already be gone: then the process is exiting anyway)
        if getattr(self, "h", None) and lib is not None:
            lib().ookd_gpu_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc, what):
        if rc != 0:
            raise OokdError(f"{what}: {lib().ookd_gpu_strerror(rc).decode()} ({lib().ookd_gpu_last_error(self.h).decode()})")

    def _result(self, res):
        # one bulk copy of the message array (56-byte records) instead of per-field ctypes access
        n = int(res.n_msgs)
        if n:
            raw = np.ctypeslib.as_array(C.cast(res.msgs, C.POINTER(C.c_uint8)), shape=(n * C.sizeof(Msg),)).copy()
            rec = raw.view(MSG_DTYPE)
        else:
            rec = np.zeros(0, dtype=MSG_DTYPE)
        msgs = msgs_to_tuples(rec, self.msg_bytes) if self.want_list else None
        return dict(msgs_raw=rec, n_in=int(res.n_in), n_out=int(res.n_out), n_buffers=int(res.n_buffers),
                    n_edges=int(res.n_edges), msgs=msgs, first_bit=int(res.first_bit),
                    sm_rounds=int(res.sm_rounds), kernel_ms=float(res.kernel_ms), fir_ms=float(res.fir_ms),
                    screen_ms=float(res.screen_ms), host_syncs=int(res.host_syncs),
                    gpu_launches=int(res.gpu_launches), refined_tiles=int(res.refined_tiles),
                    refined_blocks=int(res.refined_blocks), entry_is_provisional=int(res.entry_is_provisional),
                    entry_used=res.entry_used.astuple(), fir_mode=int(res.fir_mode))

    @property
    def halo(self):
        return int(lib().ookd_gpu_halo(self.h))

    @property
    def total_decimation(self):
        return int(lib().ookd_gpu_total_decimation(self.h))

    def decode(self, iq):
        """iq: numpy array of the handle's input format (host) or (device_ptr, n_samples)."""
        p, n, is_dev, keep = _as_ptr(iq, self.input_format)
        res = GpuResult()
        self._check(lib().ookd_gpu_decode(self.h, p, n, is_dev, C.byref(res)), "ookd_gpu_decode")
        return self._result(res)

    def decode_shard(self, iq, first_sample, n_samples, last, entry=None):
        """iq points at sample first_sample - min(halo, first_sample).  -> (result, exit carry tuple)."""
        if isinstance(iq, tuple):
            p, is_dev, keep = C.c_void_p(int(iq[0])), 1, None
        else:
            keep = _host_iq(iq, self.input_format)
            p, is_dev = C.c_void_p(keep.ctypes.data), 0
        res = GpuResult()
        ex = SmCarry()
        en = SmCarry.fromtuple(entry) if entry is not None else None
        self._check(lib().ookd_gpu_decode_shard(self.h, p, is_dev, first_sample, n_samples, int(last),
                                                C.byref(en) if en is not None else None, C.byref(ex),
                                                C.byref(res)), "ookd_gpu_decode_shard")
        return self._result(res), ex.astuple()

    def decode_begin(self, iq, first_sample, n_samples, last, entry=None):
        """First half of decode_shard: enqueue every stage and return without waiting (see ookd_gpu_decode_begin)."""
        if isinstance(iq, tuple):
            p, is_dev, keep = C.c_void_p(int(iq[0])), 1, None
        else:
            keep = _host_iq(iq, self.input_format)
            p, is_dev = C.c_void_p(keep.ctypes.data), 0
        self._keep = keep
        en = SmCarry.fromtuple(entry) if entry is not None else None
        self._check(lib().ookd_gpu_decode_begin(self.h, p, is_dev, first_sample, n_samples, int(last),
                                                C.byref(en) if en is not None else None), "ookd_gpu_decode_begin")

    def decode_end(self):
        """Second half: wait, validate, fetch the results.  -> (result, exit carry tuple)."""
        res = GpuResult()
        ex = SmCarry()
        self._check(lib().ookd_gpu_decode_end(self.h, C.byref(ex), C.byref(res)), "ookd_gpu_decode_end")
        self._keep = None
        return self._result(res), ex.astuple()

    def resolve(self, entry):
        res = GpuResult()
        ex = SmCarry()
        en = SmCarry.fromtuple(entry)
        self._check(lib().ookd_gpu_resolve(self.h, C.byref(en), C.byref(ex), C.byref(res)), "ookd_gpu_resolve")
        return self._result(res), ex.astuple()

    def edges(self):
        p = C.POINTER(C.c_uint64)()
        n = C.c_uint64()
        fb = C.c_uint32()
        self._check(lib().ookd_gpu_edges(self.h, C.byref(p), C.byref(n), C.byref(fb)), "ookd_gpu_edges")
        e = np.ctypeslib.as_array(p, shape=(n.value,)).copy() if n.value else np.zeros(0, np.uint64)
        return int(fb.value), e

    def bits(self):
        n = C.c_uint64()
        self._check(lib().ookd_gpu_bits(self.h, None, 0, C.byref(n)), "ookd_gpu_bits")
        out = np.empty(n.value, dtype=np.uint8)
        self._check(lib().ookd_gpu_bits(self.h, out.ctypes.data, n.value, C.byref(n)), "ookd_gpu_bits")
        return out

    def filtered(self, iq):
        p, n, is_dev, keep = _as_ptr(iq, self.input_format)
        m = C.c_uint64()
        self._check(lib().ookd_gpu_filtered(self.h, p, n, is_dev, None, 0, C.byref(m)), "ookd_gpu_filtered")
        out = np.empty((m.value, 2), dtype=np.float32)
        self._check(lib().ookd_gpu_filtered(self.h, p, n, is_dev, out.ctypes.data, m.value, C.byref(m)),
                    "ookd_gpu_filtered")
        return out

    def filtered_sc16q11(self):
        """Filtered samples of the last decode's shard as the reference's post-filter recorder writes them."""
        m = C.c_uint64()
        self._check(lib().ookd_gpu_filtered_sc16q11(self.h, None, 0, C.byref(m)), "ookd_gpu_filtered_sc16q11")
        out = np.empty((m.value, 2), dtype=np.int16)
        self._check(lib().ookd_gpu_filtered_sc16q11(self.h, out.ctypes.data, m.value, C.byref(m)), "ookd_gpu_filtered_sc16q11")
        return out

    def levels(self, iq, first_sample=0, n_samples=None):
        """Level histogram (include/ookd_gpu.h, "Levels") of input samples [first_sample, first_sample + n_samples):
        iq is a capture of the handle's input format pointing at sample first_sample - min(halo, first_sample), as for
        decode_shard, or (device_ptr, n) with n the samples present there.  n_samples defaults to all of them after the
        history.  -> uint64 array of LEVEL_BINS counts."""
        p, n, is_dev, keep = _as_ptr(iq, self.input_format)
        if n_samples is None:
            n_samples = n - min(self.halo, int(first_sample))
        hist = np.zeros(LEVEL_BINS, dtype=np.uint64)
        self._check(lib().ookd_gpu_levels(self.h, p, is_dev, int(first_sample), int(n_samples), hist.ctypes.data),
                    "ookd_gpu_levels")
        return hist

    def filter_cf(self, iq_f32):
        x = np.ascontiguousarray(iq_f32, dtype=np.float32).reshape(-1, 2)
        m = C.c_uint64()
        self._check(lib().ookd_gpu_filter_cf(self.h, x.ctypes.data, x.shape[0], None, 0, C.byref(m)),
                    "ookd_gpu_filter_cf")
        out = np.empty((m.value, 2), dtype=np.float32)
        self._check(lib().ookd_gpu_filter_cf(self.h, x.ctypes.data, x.shape[0], out.ctypes.data, m.value,
                                             C.byref(m)), "ookd_gpu_filter_cf")
        return out


class MultiGpu:
    """One ookd_gpu_multi handle: a window time-sharded over several GPUs of this process."""

    def __init__(self, gpu_ids, filter_stages=None, sm=None, threshold=0.1, samples_per_buffer=8192, flags=0,
                 sm_chunk_buffers=0, input_format="sc16q11", tune_step=0, deglitch=0):
        flags |= _input_format(input_format, flags)[0]
        self.input_format = input_format
        L = lib()
        cfg = GpuConfigEx()
        self._keep = []
        if filter_stages:
            fd, k = make_filter_desc(filter_stages)
            self._keep += [fd, k]
            cfg.filter = C.pointer(fd)
        if sm is not None:
            sd, k = make_sm_desc(sm["states"], sm["num_bits"], sm["sample_rate"])
            self._keep += [sd, k]
            cfg.sm = C.pointer(sd)
            self.msg_bytes = (sm["num_bits"] + 7) // 8
        else:
            self.msg_bytes = 0
        cfg.threshold = threshold
        cfg.samples_per_buffer = samples_per_buffer
        cfg.flags = flags
        cfg.sm_chunk_buffers = sm_chunk_buffers
        cfg.tune_step = tune_step
        cfg.deglitch = deglitch
        ids = (C.c_int32 * len(gpu_ids))(*gpu_ids)
        self.h = C.c_void_p()
        rc = L.ookd_gpu_multi_create(C.byref(self.h), C.byref(cfg), ids, len(gpu_ids))
        if rc != 0:
            self.h = None
            raise OokdError(f"ookd_gpu_multi_create: {L.ookd_gpu_strerror(rc).decode()}")
        self.n_gpus = len(gpu_ids)

    def close(self):
        if getattr(self, "h", None) and lib is not None:
            lib().ookd_gpu_multi_destroy(self.h)
            self.h = None

    __del__ = close

    @property
    def halo(self):
        return int(lib().ookd_gpu_multi_halo(self.h))

    def shard_range(self, first_sample, n_samples, g):
        a, b = C.c_uint64(), C.c_uint64()
        lib().ookd_gpu_multi_shard_range(self.h, first_sample, n_samples, g, C.byref(a), C.byref(b))
        return int(a.value), int(b.value)

    def decode(self, iq, first_sample=0, n_samples=None, last=True, entry=None, device_ptrs=None):
        """iq: numpy host array (the handle's input format) starting at sample first_sample - min(halo, first_sample); or device_ptrs:
        list of per-GPU device pointers.  -> (result dict, exit carry tuple)."""
        if device_ptrs is not None:
            arr = (C.c_void_p * len(device_ptrs))(*[int(p) for p in device_ptrs])
            p, is_dev, keep = C.cast(arr, C.c_void_p), 1, arr
        else:
            keep = _host_iq(iq, self.input_format)
            p, is_dev = C.c_void_p(keep.ctypes.data), 0
            if n_samples is None:
                n_samples = keep.size // 2 - min(self.halo, first_sample)
        res = GpuResult()
        ex = SmCarry()
        en = SmCarry.fromtuple(entry) if entry is not None else None
        rc = lib().ookd_gpu_multi_decode(self.h, p, is_dev, first_sample, n_samples, int(last),
                                         C.byref(en) if en is not None else None, C.byref(ex), C.byref(res))
        if rc != 0:
            raise OokdError(f"ookd_gpu_multi_decode: {lib().ookd_gpu_strerror(rc).decode()} "
                            f"({lib().ookd_gpu_multi_last_error(self.h).decode()})")
        n = int(res.n_msgs)
        if n:
            raw = np.ctypeslib.as_array(C.cast(res.msgs, C.POINTER(C.c_uint8)), shape=(n * C.sizeof(Msg),)).copy()
            rec = raw.view(MSG_DTYPE)
        else:
            rec = np.zeros(0, dtype=MSG_DTYPE)
        return dict(msgs_raw=rec, msgs=msgs_to_tuples(rec, self.msg_bytes), n_in=int(res.n_in), n_out=int(res.n_out),
                    n_buffers=int(res.n_buffers), n_edges=int(res.n_edges), first_bit=int(res.first_bit),
                    sm_rounds=int(res.sm_rounds), kernel_ms=float(res.kernel_ms), gpu_launches=int(res.gpu_launches),
                    shards_used=int(lib().ookd_gpu_multi_shards_used(self.h))), ex.astuple()

    def edges(self):
        p = C.POINTER(C.c_uint64)()
        n = C.c_uint64()
        fb = C.c_uint32()
        rc = lib().ookd_gpu_multi_edges(self.h, C.byref(p), C.byref(n), C.byref(fb))
        if rc != 0:
            raise OokdError(f"ookd_gpu_multi_edges: {lib().ookd_gpu_multi_last_error(self.h).decode()}")
        e = np.ctypeslib.as_array(p, shape=(n.value,)).copy() if n.value else np.zeros(0, np.uint64)
        return int(fb.value), e


def synth(n_samples, toggles, i_on, q_on, noise_scale, seed, first_sample=0, device_id=-1, device_ptr=None,
          noise_terms=4):
    """Synthetic capture on the GPU.  Returns numpy (n,2) int16, or fills device_ptr when given."""
    tg = np.ascontiguousarray(toggles, dtype=np.uint64)
    if device_ptr is not None:
        rc = lib().ookd_gpu_synth_ex(device_id, C.c_void_p(int(device_ptr)), 1, first_sample, n_samples,
                                     tg.ctypes.data, len(tg), int(i_on), int(q_on), int(noise_scale), int(seed),
                                     int(noise_terms))
        out = None
    else:
        out = np.empty((n_samples, 2), dtype=np.int16)
        rc = lib().ookd_gpu_synth_ex(device_id, out.ctypes.data, 0, first_sample, n_samples, tg.ctypes.data, len(tg),
                                     int(i_on), int(q_on), int(noise_scale), int(seed), int(noise_terms))
    if rc != 0:
        raise OokdError(f"ookd_gpu_synth: {lib().ookd_gpu_strerror(rc).decode()}")
    return out


def batch_decode(gpus, captures, msgs_cap=None):
    """Independent captures through ookd_gpu_batch_decode.  gpus: list of Gpu handles; captures: list of
    (iq, handle_index) with iq a numpy array in the input format of gpus[handle_index] (host) or (device_ptr, n_samples).
    -> list of structured message arrays (MSG_DTYPE), one per capture, plus the per-capture statistics."""
    n = len(captures)
    caps = (Capture * max(n, 1))()
    keep = []
    for i, (iq, hi) in enumerate(captures):
        if isinstance(iq, tuple):
            caps[i].iq, caps[i].n_samples, caps[i].iq_is_device_ptr = int(iq[0]), int(iq[1]), 1
        else:
            a = _host_iq(iq, gpus[hi].input_format)
            keep.append(a)
            caps[i].iq, caps[i].n_samples, caps[i].iq_is_device_ptr = a.ctypes.data, a.size // 2, 0
        caps[i].handle = hi
    handles = (C.c_void_p * len(gpus))(*[g.h for g in gpus])
    first = (C.c_uint64 * (n + 1))()
    results = (GpuResult * max(n, 1))()
    # (a list that does not fit costs a SECOND decode of the whole batch: start with room for 256 messages per capture)
    cap = int(msgs_cap) if msgs_cap is not None else max(4096, 256 * n)
    while True:
        out = np.zeros(cap, dtype=MSG_DTYPE)
        rc = lib().ookd_gpu_batch_decode(handles, len(gpus), caps, n, out.ctypes.data, cap, first, results)
        if rc == -5 and msgs_cap is None and first[n] > cap:       # OOKD_ERR_OVERFLOW: decode again with room for all
            cap = int(first[n])
            continue
        if rc != 0:
            raise OokdError(f"ookd_gpu_batch_decode: {lib().ookd_gpu_strerror(rc).decode()}")
        break
    msgs = [out[first[i]:first[i + 1]].copy() for i in range(n)]
    stats = [dict(n_in=int(results[i].n_in), n_edges=int(results[i].n_edges), kernel_ms=float(results[i].kernel_ms),
                  host_syncs=int(results[i].host_syncs), gpu_launches=int(results[i].gpu_launches)) for i in range(n)]
    return msgs, stats
