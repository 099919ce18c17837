"""TEST INFRASTRUCTURE: recorded comparisons with the reference, so that the tests comparing with it run without it.

A test that steps the product (or the C oracle) beside the reference compares, check after check, a value of the
reference with the product's.  A Tape stands for the reference side of those comparisons:

  * recording (AIE_RECORD_REFERENCE=1 where the reference can run): the comparisons run against the live reference
    exactly as before, and the reference's values are also recorded per test case under tests/golden/reference_tapes/;
  * replaying (everywhere else): the reference is not imported and the product's values are checked against the record.

What is recorded, per test case:
  * exact comparisons (`equal`): a SHA-1 over every checked value in order, so any difference in any checked value fails;
    a 16-bit checkpoint of it every CHECKPOINT checks tells where a replay first diverged;
  * comparisons with a tolerance (`close`, `metric`):
      - the reference's values themselves for every STRIDE-th check of each key (the phase taken from the key, so the
        sampled steps differ between keys), stored in tests/golden/reference_tapes/<family>.npz and compared element by
        element with the original tolerance;
      - for every check, two projections of the reference's values, summed per quantity (the key with agent indices
        dropped): one with +-1 weights drawn from the full key, the check's index within that key and the element's
        position (values moved between agents, steps or positions change it), one with the signs of the product's values
        (a systematic relative error of the order of the tolerance changes it).  Where every element is within the
        tolerance, the product's sums differ from them by at most the summed tolerance, so replay never fails a run that
        the live comparison passes; a larger difference fails.
    Sizes, NaN / inf positions and the set of quantities go into the SHA-1.
The digests are computed in float64 on values cast the way the live comparisons see them (np.array_equal / np.allclose
compare values, not dtypes or shapes: shapes are flattened unless asked for, -0.0 equals 0.0).
"""
import contextlib
import hashlib
import json
import lzma
import os
import re
import zlib

import numpy as np

from oracle import ref_harness as rh

TAPE_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_tapes")
CHECKPOINT = 256
STRIDE = 16
_FILES = {}
_VALUES = {}


class Mismatch(AssertionError):
    """A compared value differs from the reference (live) or from its recorded digest (replay)."""


class Refused(Exception):
    """The reference refused the configuration of the case (recorded, so that replay skips the case as live runs did)."""


def _check(ok, msg):
    if not ok:
        raise Mismatch(msg)


def recording():
    return os.environ.get("AIE_RECORD_REFERENCE", "0") not in ("", "0")


def _weights(key, i, n):
    """+-1 per element, from the full key, the check's index within the key and the element's position."""
    x = np.arange(n, dtype=np.uint32) * np.uint32(0x9E3779B1) ^ np.uint32(zlib.crc32(("%s\0%d" % (key, i)).encode()))
    x ^= x >> np.uint32(16)
    x *= np.uint32(0x85EBCA6B)
    x ^= x >> np.uint32(13)
    return np.where(x >> np.uint32(15) & np.uint32(1), 1.0, -1.0)


def _quantity(key):
    """The key with agent / bracket indices dropped: per-agent values of one quantity share a projection."""
    return re.sub(r"(^|/)\d+(?=/|$|\[)", r"\1#", key)


def _values(x):
    """float64 vector of a value as np.array_equal sees it (strings and name lists hash their text)."""
    if isinstance(x, str):
        return None, x.encode()
    if isinstance(x, (list, tuple, set, frozenset)) and x and all(isinstance(v, str) for v in x):
        return None, "\0".join(sorted(x) if isinstance(x, (set, frozenset)) else x).encode()
    v = np.asarray(x, np.float64).ravel() + 0.0   # + 0.0: -0.0 -> 0.0
    return v, None


def _load(family):
    if family not in _FILES:
        p = os.path.join(TAPE_DIR, family + ".json")
        _FILES[family] = json.load(open(p)) if os.path.exists(p) else {}
    return _FILES[family]


def _load_values(family):
    """{case: {"flags" | "f32" | "f64": lzma-compressed bytes}}: the sampled reference values of a family."""
    if family not in _VALUES:
        p = os.path.join(TAPE_DIR, family + ".npz")
        _VALUES[family] = {}
        if os.path.exists(p):
            with np.load(p) as z:
                for name in z.files:
                    case, part = name.rsplit(":", 1)
                    _VALUES[family].setdefault(case, {})[part] = z[name]
    return _VALUES[family]


def _save(family):
    os.makedirs(TAPE_DIR, exist_ok=True)
    data = _FILES[family]
    with open(os.path.join(TAPE_DIR, family + ".json"), "w") as f:
        f.write("{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(data[k], sort_keys=True)) for k in sorted(data))
                + "\n}\n")
    values = {"%s:%s" % (case, part): a for case, parts in _load_values(family).items() if case in data
              for part, a in parts.items()}
    if values:
        np.savez(os.path.join(TAPE_DIR, family + ".npz"), **values)


def _pack(words):
    return np.frombuffer(lzma.compress(b"".join(w.tobytes() for w in words), preset=9), np.uint8)


def _unpack(blob, dtype):
    return np.frombuffer(lzma.decompress(blob.tobytes()), dtype)


class Tape:
    """The reference side of one test case.  `live` is True while recording: the caller then runs the reference and passes
    its values as `want`; while replaying `want` is ignored (pass None) and the recorded digests stand in for it."""

    def __init__(self, family=None, case=None, available=rh.reference_available):
        """family None: live comparisons only, nothing stored (the fuzz tools).  available: whether the reference side can
        run here (default: the reference tree is importable)."""
        self.family, self.case = family, str(case)
        self.live = family is None or recording()
        if self.live and not available():
            raise RuntimeError("comparing with the live reference needs it here (reference tree: %s)" % rh.REFERENCE_ROOT)
        self.n, self.sha, self.marks, self.proj, self.slack, self.sites = 0, hashlib.sha1(), [], {}, {}, {}
        self.occ, self.prev, self.flags, self.words = {}, {}, [], {np.uint32: [], np.uint64: []}
        if not self.live:
            rec = _load(family).get(self.case)
            if rec is not None and "refused" in rec:
                raise Refused(rec["refused"])
            _check(rec is not None, "no recorded reference for %s/%s: record it with AIE_RECORD_REFERENCE=1" % (family, case))
            self.rec = rec
            v = _load_values(family).get(self.case, {})
            self.flags = _unpack(v["flags"], np.uint8) if "flags" in v else np.zeros(0, np.uint8)
            self.words = {t: _unpack(v[part], t) if part in v else np.zeros(0, t) for t, part in ((np.uint32, "f32"), (np.uint64, "f64"))}
            self.cursor = {np.uint32: 0, np.uint64: 0, np.uint8: 0}

    # ---- exact ------------------------------------------------------------------------------------------------------
    def _key(self, key, want, got, shape):
        """shape=True: the shapes must agree as well (folded into the key)."""
        if not shape:
            return key
        if self.live:
            _check(np.shape(want) == np.shape(got), "%s: shape %s vs %s" % (key, np.shape(want), np.shape(got)))
        return "%s%s" % (key, np.shape(got))

    def equal(self, key, want, got, where="", shape=False):
        """np.array_equal(want, got) on the flattened values (names and strings: equal text)."""
        key = self._key(key, want, got, shape)
        (wv, wt), (gv, gt) = (_values(want) if self.live else (None, None)), _values(got)
        if self.live:
            _check((wt == gt) if wv is None else (gv is not None and np.array_equal(wv, gv)), "%s %s" % (where, key))
        v, text = (wv, wt) if self.live else (gv, gt)
        self.sha.update(key.encode() + b"\0" + (text if v is None else np.isnan(v).tobytes() + np.nan_to_num(v).tobytes()))
        self.n += 1
        if self.n % CHECKPOINT == 0:
            mark = self.sha.hexdigest()[:4]
            if self.live:
                self.marks.append(mark)
            else:
                i = 4 * (self.n // CHECKPOINT - 1)
                _check(self.rec["marks"][i:i + 4] == mark,
                       "%s %s: differs from the recorded reference within checks %d..%d" % (where, key, self.n - CHECKPOINT, self.n))

    # ---- with a tolerance -------------------------------------------------------------------------------------------
    def close(self, key, want, got, rtol, atol, where="", shape=False, equal_nan=False):
        """np.allclose(want, got, rtol, atol): |want - got| <= atol + rtol * |got| element by element."""
        key = self._key(key, want, got, shape)
        g = np.asarray(got, np.float64).ravel()
        if self.live:
            w = np.asarray(want, np.float64).ravel()
            _check(w.size == g.size and np.allclose(w, g, rtol=rtol, atol=atol, equal_nan=equal_nan), "%s %s" % (where, key))
        i = self._sample(key, w if self.live else None, g, lambda w: np.isclose(w, g, rtol=rtol, atol=atol, equal_nan=equal_nan), where)
        self._fold_close(key, i, w if self.live else g, g, atol + rtol * np.abs(g))

    def metric(self, key, want, got, where=""):
        """metric values: equal NaN-ness, |want - got| <= 1e-6 * max(1, |want|)."""
        b = float(got)
        if self.live:
            a = float(want)
            _check((np.isnan(a) and np.isnan(b)) or abs(a - b) <= 1e-6 * max(1.0, abs(a)),
                   "%s metric %s: %r vs %r" % (where, key, a, b))
        v = np.array([float(want) if self.live else b])
        i = self._sample(key, v if self.live else None, np.array([b]),
                         lambda a: (np.isnan(a) & np.isnan(b)) | (np.abs(a - b) <= 1e-6 * np.maximum(1.0, np.abs(a))), where)
        # |want| <= |got| + 1e-6 max(1, |want|): the bound in terms of got, for replay
        self._fold_close(key, i, v, np.array([b]), np.array([1.000002e-6 * max(1.0, abs(b) / (1 - 1e-6))]))

    def _sample(self, key, w, g, ok, where):
        """Counts the check within its key; for every STRIDE-th one, stores the reference's values w (recording) or compares
        g with the stored ones element by element, ok(stored) being the live comparison (replay).  Returns the index."""
        i = self.occ.get(key, 0)
        self.occ[key] = i + 1
        if self.family is None or (i + zlib.crc32(key.encode())) % STRIDE:
            return i
        if self.live:
            w = np.ascontiguousarray(w, np.float64)
            f32 = bool(np.array_equal(w.astype(np.float32).astype(np.float64), w, equal_nan=True))
            bits = w.astype(np.float32).view(np.uint32) if f32 else w.view(np.uint64)
            self.flags.append(np.uint8(f32))
        else:
            _check(self.cursor[np.uint8] < self.flags.size, "%s %s: more sampled checks than recorded" % (where, key))
            f32 = bool(self.flags[self.cursor[np.uint8]])
            self.cursor[np.uint8] += 1
            t = np.uint32 if f32 else np.uint64
            c = self.cursor[t]
            bits = self.words[t][c:c + g.size]
            _check(bits.size == g.size, "%s %s: recorded values exhausted" % (where, key))
            self.cursor[t] = c + g.size
        prev = self.prev.get(key)
        delta = prev is not None and prev.dtype == bits.dtype and prev.size == bits.size   # stored as XOR with the last sample
        if self.live:
            self.words[np.uint32 if f32 else np.uint64].append(bits ^ prev if delta else bits)
        else:
            bits = bits ^ prev if delta else bits
            stored = bits.view(np.float32 if f32 else np.float64).astype(np.float64)
            bad = np.flatnonzero(~ok(stored))
            _check(bad.size == 0, "%s %s: element %s is %r, the reference's %r" % (
                where, key, bad[:1].tolist(), g[bad[:1]].tolist(), stored[bad[:1]].tolist()))
        self.prev[key] = bits
        return i

    def _fold_close(self, key, i, v, g, tol):
        """i: the check's index within its key; v: the values folded (the reference's recording, the product's replaying);
        g: the product's values."""
        fin = np.isfinite(v)
        kind = np.where(np.isnan(v), 1, np.where(v == np.inf, 2, np.where(v == -np.inf, 3, 0))).astype(np.int8)
        self.sha.update(("%s\0%d\0" % (key, v.size)).encode() + kind.tobytes())
        v = np.where(fin, v, 0.0)   # NaN / inf must match exactly (above); finite values within the tolerance
        q = _quantity(key)
        self.proj[q] = self.proj.get(q, 0.0) + np.array([_weights(key, i, v.size) @ v, np.sign(np.where(np.isfinite(g), g, 0.0)) @ v])
        self.slack[q] = self.slack.get(q, 0.0) + float(np.sum(tol[fin])) + 1e-12 * float(np.sum(np.abs(v)))

    # ---- structure ---------------------------------------------------------------------------------------------------
    def keys(self, site, candidates, present=()):
        """The candidates the reference offered (`present`, recording) at a comparison site, recorded once per site as a
        bit mask over `candidates`; replay returns the recorded selection."""
        candidates = list(candidates)
        if self.live:
            mask = sum(1 << i for i, k in enumerate(candidates) if k in present)
            _check(self.sites.setdefault(site, mask) == mask, "%s: keys changed" % site)
        else:
            mask = self.rec["sites"][site]
        return [k for i, k in enumerate(candidates) if mask >> i & 1]

    @contextlib.contextmanager
    def refusals(self, errors, when=lambda ex: True):
        """Live: an exception of `errors` (but no Mismatch) for which when(ex) holds is the reference refusing the case's
        configuration; it is recorded and raised as Refused.  Replay: nothing to catch (a recorded refusal raises Refused
        when the Tape is made)."""
        if not self.live:
            yield
            return
        try:
            yield
        except errors as ex:
            if isinstance(ex, Mismatch) or not when(ex):
                raise
            if self.family is not None:
                _load(self.family)[self.case] = {"refused": repr(ex)[:300]}
                _save(self.family)
            raise Refused(repr(ex)) from ex

    def finish(self):
        """Store (recording) or check (replay) the digests of the whole case."""
        if self.family is None:
            return
        quantities = sorted(self.proj)
        self.sha.update("\0".join(quantities).encode())
        if self.live:   # 10 significant digits: the rounding (<= 1e-9 relative) is added to the tolerance on replay
            _load(self.family)[self.case] = {
                "checks": self.n, "sha1": self.sha.hexdigest(), "marks": "".join(self.marks), "sites": self.sites,
                "close": [float("%.10g" % x) for q in quantities for x in self.proj[q]]}
            parts = {"flags": [np.array(self.flags, np.uint8)], "f32": self.words[np.uint32], "f64": self.words[np.uint64]}
            _load_values(self.family)[self.case] = {k: _pack(v) for k, v in parts.items() if sum(w.size for w in v)}
            _save(self.family)
            return
        rec = self.rec
        _check(self.n == rec["checks"], "%d exact checks, %d recorded" % (self.n, rec["checks"]))
        _check(self.cursor[np.uint8] == self.flags.size, "fewer sampled checks than recorded")
        _check(2 * len(quantities) == len(rec["close"]), "%d compared quantities, %d recorded" % (len(quantities), len(rec["close"]) // 2))
        for q, want in zip(quantities, np.reshape(rec["close"], (-1, 2))):
            d = np.abs(self.proj[q] - want)
            _check(np.all(d <= self.slack[q] + 1e-9 * np.abs(want)),
                   "%s: differs from the recorded reference by %s (tolerance %g)" % (q, d, self.slack[q]))
        _check(self.sha.hexdigest() == rec["sha1"], "exact checks differ from the recorded reference")


def flags(done):
    """A done dictionary as text, for `equal`."""
    return ["%s=%d" % (k, bool(v)) for k, v in sorted(done.items())]


def same_tree(tape, key, want, got, where="", rtol=1e-6, atol=1e-7):
    """Nested dictionaries (observations, rewards): the same keys, leaves within the tolerance.  `key` names the place in
    the tree for the digests, `where` (the step) only goes into messages."""
    if isinstance(got, dict) or (tape.live and isinstance(want, dict)):
        tape.equal(key + "/", sorted(map(str, want)) if tape.live else None, sorted(map(str, got)) if isinstance(got, dict) else [], where)
        for k in sorted(got, key=str):
            same_tree(tape, "%s/%s" % (key, k), want[k] if tape.live else None, got[k], where, rtol, atol)
    else:
        tape.close(key, want, got, rtol, atol, where)


def same_log(tape, key, want, got, where=""):
    """A dense log (JSON structure): the same keys and lengths, equal strings, numbers within 1e-6 relative; a None of
    the reference matches None or NaN."""
    live = tape.live
    if isinstance(got, dict) or (live and isinstance(want, dict)):
        tape.equal(key + "/", sorted(map(str, want)) if live else None, sorted(map(str, got)) if isinstance(got, dict) else [], where)
        for k in sorted(got, key=str):
            same_log(tape, "%s/%s" % (key, k), want[k] if live else None, got[k], where)
    elif isinstance(got, (list, tuple)) or (live and isinstance(want, list)):
        tape.equal(key + "#", len(want) if live else None, len(got) if isinstance(got, (list, tuple)) else -1, where)
        for i, g in enumerate(got):
            same_log(tape, key + "[]", want[i] if live else None, g, where)
    elif isinstance(got, str) or (live and isinstance(want, str)):
        tape.equal(key, want, got, where)
    else:
        tape.metric(key, float("nan") if want is None else want, float("nan") if got is None else got, where)


def same_metrics(tape, key, want, got, where=""):
    """env.metrics-like flat dictionaries: the same keys, values within 1e-6 relative (NaN matches NaN)."""
    tape.equal(key + "/", sorted(want) if tape.live else None, sorted(got), where)
    for k in sorted(got):
        tape.metric("%s/%s" % (key, k), want[k] if tape.live else None, got[k], where)
