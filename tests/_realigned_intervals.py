"""numpy restatement of `with_tracks(kind="realigned-intervals")` (DESIGN.md §7): the walk of the reference's
shift_and_realign_track_core (src/tracks/mod.rs:224-406, restated in C by the oracle) with PROVENANCE instead of values --
every output position records where its value comes from -- then the maximal runs of one identity other than none.

Identities: a source position s in [0, track_n) is the index of the stored interval that holds q_start + s (none if no
interval does, or outside [0, track_n)); Repeat5pNormalized and Constant fills are one identity per variant; FlankSample
positions take the identity of the position they sample; Interpolate positions are one identity each."""
import numpy as np

REPEAT_5P, REPEAT_5P_NORM, CONSTANT, FLANK_SAMPLE, INTERPOLATE = range(5)
_M64 = (1 << 64) - 1


def xorshift64(x: int) -> int:
    x ^= (x << 13) & _M64
    x ^= x >> 7
    x ^= (x << 17) & _M64
    return x


def hash4(a: int, b: int, c: int, d: int) -> int:
    h = xorshift64(a ^ b)
    h = xorshift64(h ^ c)
    return xorshift64(h ^ d)


class Slot:
    """The stored intervals of one slot (sorted, free of overlaps) seen from a window that starts at q_start."""

    def __init__(self, starts, ends, values, q_start: int, track_n: int):
        self.s = np.asarray(starts, np.int64)
        self.e = np.asarray(ends, np.int64)
        self.v = np.asarray(values, np.float32)
        self.q_start, self.track_n = int(q_start), int(track_n)

    def ident(self, s: int):
        """Index of the interval that holds relative source position s, or None."""
        if s < 0 or s >= self.track_n:
            return None
        g = self.q_start + s
        i = int(np.searchsorted(self.s, g, side="right")) - 1
        return i if i >= 0 and self.e[i] > g else None

    def value(self, s: int) -> np.float32:
        i = self.ident(s)
        return self.v[i] if i is not None else np.float32(0.0)


def _lagrange(slot: Slot, k: int, v_len: int, v_rel_pos: int, i: int) -> np.float32:
    xs = [-float(j) for j in range(k)] + [float(v_len) + float(j) for j in range(k)]
    ys = [float(slot.value(max(v_rel_pos - j, 0))) for j in range(k)]
    ys += [float(slot.value(min(v_rel_pos + 1 + j, slot.track_n - 1))) for j in range(k)]
    x, acc = float(i), 0.0
    for a in range(2 * k):
        term = ys[a]
        for b in range(2 * k):
            if b != a:
                term *= (x - xs[b]) / (xs[a] - xs[b])
        acc += term
    return np.float32(acc)


def provenance(var_starts, var_ilens, keep, shift: int, slot: Slot, length: int, strategy: int, param: float,
               base_seed: int, query: int, hap: int):
    """Per output position of one realigned row: (identity, float32 value).  Identities are ("s", interval index),
    ("v", variant), ("p", position) or None."""
    ident = [None] * length
    value = [np.float32(0.0)] * length

    def src(o, s):
        i = slot.ident(s)
        ident[o] = ("s", i) if i is not None else None
        value[o] = slot.v[i] if i is not None else np.float32(0.0)

    n = len(var_starts)
    if n == 0:  # :240-246
        for o in range(length):
            src(o, o)
        return ident, value
    track_idx = out_idx = shifted = 0
    for v in range(n):
        if keep is not None and not keep[v]:
            continue
        v_diff = int(var_ilens[v])
        v_rel_pos = int(var_starts[v]) - slot.q_start
        v_rel_end = v_rel_pos - min(v_diff, 0) + 1
        if v_diff < 0 and v_rel_pos < 0 and v_rel_end >= 0:
            track_idx = v_rel_end
            continue
        if v_rel_pos < track_idx:
            continue
        v_len = max(v_diff, 0) + 1
        if shifted < shift:
            dist = v_rel_pos - track_idx
            if shifted + dist + v_len < shift:
                continue
            elif shifted + dist >= shift:
                track_idx += shift - shifted
                shifted = shift
            else:
                a = shift - shifted - dist
                shifted = shift
                if a == v_len:
                    track_idx = v_rel_end
                    continue
                track_idx = v_rel_pos
                v_len -= a
        if v_diff == 0:
            continue
        track_len = v_rel_pos - track_idx
        if out_idx + track_len >= length:
            break
        for i in range(track_len):
            src(out_idx + i, track_idx + i)
        out_idx += track_len
        w = min(v_len, length - out_idx)
        if v_diff > 0 and strategy != REPEAT_5P:
            for i in range(w):
                o = out_idx + i
                if strategy == REPEAT_5P_NORM:
                    ident[o], value[o] = ("v", v), np.float32(slot.value(v_rel_pos) / np.float32(v_len))
                elif strategy == CONSTANT:
                    ident[o], value[o] = ("v", v), np.float32(param)
                elif strategy == FLANK_SAMPLE:
                    width = int(param)
                    lo, hi = max(v_rel_pos - width, 0), min(v_rel_pos + width, slot.track_n - 1)
                    size = (hi - lo + 1) & _M64
                    src(o, lo + hash4(base_seed, query, hap, o) % size)
                else:
                    k = (int(param) + 2) // 2
                    ident[o], value[o] = ("p", o), _lagrange(slot, k, v_len, v_rel_pos, i)
        else:
            for i in range(w):
                src(out_idx + i, v_rel_pos)
        out_idx += w
        track_idx = v_rel_end
        if out_idx >= length:
            break
    if shifted < shift:
        track_idx = min(track_idx + shift - shifted, slot.track_n)
    rest = length - out_idx
    if rest > 0:
        for i in range(max(min(rest, slot.track_n - track_idx), 0)):
            src(out_idx + i, track_idx + i)
    return ident, value


def runs(ident, value, w0: int):
    """The maximal runs of one identity other than None -> (starts, ends, values float32), haplotype coordinates from w0."""
    s, e, v = [], [], []
    o, n = 0, len(ident)
    while o < n:
        if ident[o] is None:
            o += 1
            continue
        b = o
        while b + 1 < n and ident[b + 1] == ident[o]:
            b += 1
        s.append(w0 + o)
        e.append(w0 + b + 1)
        v.append(value[o])
        o = b + 1
    return np.asarray(s, np.int32), np.asarray(e, np.int32), np.asarray(v, np.float32)


def realigned_intervals_row(var_starts, var_ilens, keep, shift, slot: Slot, length, strategy=REPEAT_5P, param=0.0, base_seed=0,
                            query=0, hap=0):
    """One row's intervals (starts, ends, values float32), coordinates from the slot's q_start."""
    ident, value = provenance(var_starts, var_ilens, keep, shift, slot, length, strategy, param, base_seed, query, hap)
    return runs(ident, value, slot.q_start)


def paint(starts, ends, values, w0: int, length: int, rc: bool = False) -> np.ndarray:
    """Intervals painted into zeros of `length` from w0, reversed when `rc`."""
    out = np.zeros(length, np.float32)
    for a, b, v in zip(starts, ends, values):
        out[int(a) - w0:int(b) - w0] = v
    return out[::-1].copy() if rc else out
