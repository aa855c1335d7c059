"""CPU restatements of the deglitch vote (include/ookd_gpu.h, "Deglitch"), written independently of the GPU's word
method:

- vote(): the whole decision string at once, a convolution with ones(2M+1) over 2M leading zeros, >= M+1;
- StreamVote: buffer by buffer, as a receiver would run it, carrying the last 2M raw decisions and their count;
- rx(): the oracle's receive loop with the streaming vote between the threshold and everything that consumes
  decisions (edges, first_bit, the state machine, per samples_per_buffer buffer as ookd_oracle_rx drives it).

The oracle itself restates the reference program, which has no vote, so this lives with the tests."""
import numpy as np

from oracle import oracle as O


def vote(bits, m):
    """v(i) = [r(i-2M) + ... + r(i) >= M+1], r = 0 before output 0."""
    bits = np.asarray(bits, dtype=np.uint8)
    if m == 0 or bits.size == 0:                   # (np.convolve swaps its arguments when the first is shorter)
        return bits.copy()
    r = np.concatenate([np.zeros(2 * m, np.int64), bits.astype(np.int64)])
    c = np.convolve(r, np.ones(2 * m + 1, np.int64), mode="valid")
    return (c >= m + 1).astype(np.uint8)


class StreamVote:
    """The vote over a stream cut into pieces of any length: a ring of the last 2M raw decisions and their count."""

    def __init__(self, m):
        self.m = m
        self.ring = np.zeros(2 * m, np.uint8)      # raw decisions before the next piece, oldest first
        self.count = 0                             # = ring.sum()

    def push(self, raw):
        raw = np.asarray(raw, dtype=np.uint8)
        m, n = self.m, raw.size
        if m == 0 or n == 0:
            return raw.copy()
        x = np.concatenate([self.ring, raw]).astype(np.int64)
        # count of the 2M decisions before output i of the piece: the carried count, plus what entered since the piece
        # began, minus what left
        entered = np.concatenate([[0], np.cumsum(x[2 * m:2 * m + n - 1])])
        left = np.concatenate([[0], np.cumsum(x[:n - 1])])
        before = self.count + entered - left
        out = (before + raw >= m + 1).astype(np.uint8)
        self.ring = x[n:].astype(np.uint8)
        self.count = int(before[-1] + raw[-1] - x[n - 1])
        assert self.count == int(self.ring.sum())
        return out


def rx(iq, filter_stages, device, threshold_=0.1, samples_per_buffer=8192, samplerate=3000000, deglitch=0):
    """O.rx with the vote: -> dict(n_out, n_buffers, first_bit, edges, msgs, bits (voted), raw_bits)."""
    ref = O.rx(iq, filter_stages, None, threshold_=threshold_, samples_per_buffer=samples_per_buffer,
               samplerate=samplerate, want_bits=True)
    raw = ref["bits"]
    dec = O.filter_total_decimation(filter_stages) if filter_stages else 1
    sm = O.Sm(device, samplerate // dec) if device else None
    sv = StreamVote(deglitch)
    voted = np.empty_like(raw)
    msgs = []
    lo = 0
    for b in range(ref["n_buffers"]):
        hi = min(((b + 1) * samples_per_buffer) // dec, raw.size)   # outputs whose last input lies in buffers 0..b
        buf = sv.push(raw[lo:hi])
        voted[lo:hi] = buf
        if sm is not None:                                          # device_process, src/device.c:634-658
            total, r = 0, 0
            while total < buf.size and r != -1:
                r, n = sm.process(buf[total:])
                total += n
                if r == 1:
                    msgs.append((lo + total - 1, b, sm.get_state()[2], sm.data()))
        lo = hi
    assert lo == raw.size
    edges = (np.flatnonzero(voted[1:] != voted[:-1]) + 1).astype(np.uint64)
    return dict(n_out=ref["n_out"], n_buffers=ref["n_buffers"], first_bit=int(voted[0]) if voted.size else 0,
                edges=edges, msgs=msgs, bits=voted, raw_bits=raw)
