"""The original project's CPU path (oracle/ref.py) as the tests see it, replayed from stored outputs.

Every array a test takes from the reference is stored as a fixed, seeded sample of its elements, spread over its rows
(plus every non-finite element, the first eight, the last of every row and the largest magnitude of every row), in
tests/golden/reference_outputs.{json,npz}, keyed by test id and call order, with a crc32 of the inputs the test had handed
to the reference up to that call (a replay whose inputs differ warns that the outputs need recording again). `Reference` has the call surface of oracle/ref.py: by default it replays those samples, so the comparisons run
where the original project is absent; with B200_RECORD_REFERENCE=1, where oracle/_ref/libjst_ref.so exists, it runs the
real reference and rewrites the stored samples at the end of the session (run the whole suite, GPU tests included).

A test compares its own full result against a `Sample` with `sample.take(got)` / `sample.values`, or hands the sample to
tests/parity.py, whose checks accept one in place of the full array.
"""
from __future__ import annotations

import json
import os
import warnings
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
JSON_PATH = os.path.join(HERE, "golden", "reference_outputs.json")
NPZ_PATH = os.path.join(HERE, "golden", "reference_outputs.npz")
SAMPLES = 44                  # random elements kept per output array, spread over its rows (all when it is smaller)
MAX_ROWS = 64                 # outputs with more rows keep one overall maximum and last element instead of one per row
RECORD = bool(os.environ.get("B200_RECORD_REFERENCE"))


def _crc(crc: int, value) -> int:
    """crc32 of what a test hands the reference: arrays by dtype, shape and bytes, other values by repr. Reference
    outputs fed back (`Sample`) are left out: only their recording has the whole array."""
    if isinstance(value, Sample):
        return crc
    if isinstance(value, np.ndarray):
        a = np.ascontiguousarray(value)
        return zlib.crc32(a.tobytes(), zlib.crc32(f"{a.dtype.str}{a.shape}".encode(), crc))
    if isinstance(value, dict):
        for k in sorted(value, key=str):
            crc = _crc(_crc(crc, k), value[k])
        return crc
    if isinstance(value, (list, tuple)):
        for v in value:
            crc = _crc(crc, v)
        return crc
    return zlib.crc32(repr(value).encode(), crc)


class RefError(RuntimeError):
    """A call the reference refused (its error message is stored and raised again on replay)."""


class Sample:
    """The stored part of one reference output: shape and dtype, the values at flat indices `idx`, and the largest
    finite magnitude of every row (last axis; of the whole array when it has more than MAX_ROWS rows)."""

    def __init__(self, shape, dtype, idx, values, row_absmax, full=None):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        self.idx, self.values, self.row_absmax = idx, values, row_absmax
        self.full = full              # the whole output while recording (to feed a later reference stage), else None

    @classmethod
    def of(cls, key: str, full: np.ndarray) -> "Sample":
        flat = full.reshape(-1)
        n = flat.size
        rng = np.random.default_rng(zlib.crc32(key.encode()))
        picks = [np.flatnonzero(~np.isfinite(flat)), np.arange(min(n, 8))]     # first eight: hand-set edge values
        all_rows = int(np.prod(full.shape[:-1])) if full.ndim > 1 and full.shape[-1] else 1
        if n > SAMPLES:
            # SAMPLES elements spread over the rows (every row gets some while there are fewer rows than samples)
            length = n // all_rows
            row = np.arange(SAMPLES) % all_rows if all_rows <= SAMPLES else rng.choice(all_rows, SAMPLES, replace=False)
            picks.append(row * length + rng.integers(0, length, SAMPLES))
        else:
            picks.append(np.arange(n))
        # the last element and the largest magnitude of every row (one row when there are more than MAX_ROWS)
        rows = all_rows if all_rows <= MAX_ROWS else 1
        mag = np.where(np.isfinite(flat), np.abs(flat), -1.0).reshape(rows, -1)
        if mag.size:
            picks.append(np.arange(1, rows + 1) * mag.shape[1] - 1)
            picks.append(mag.argmax(axis=1) + np.arange(rows) * mag.shape[1])
        row_absmax = np.maximum(mag.max(axis=1, initial=-1.0), 0.0).astype(np.float32)
        idx = np.unique(np.concatenate(picks)).astype(np.int64)
        return cls(full.shape, full.dtype, idx, flat[idx].copy(), row_absmax, full)

    @property
    def size(self) -> int:
        return int(np.prod(self.shape))

    def array(self) -> np.ndarray:
        """The whole output; only for outputs small enough to be stored whole."""
        assert self.idx.size == self.size, f"only {self.idx.size} of {self.size} elements are stored"
        return self.values.reshape(self.shape)

    def take(self, a) -> np.ndarray:
        """The elements of a full array of this shape at the stored positions."""
        a = np.asarray(a)
        assert a.shape == self.shape, (a.shape, self.shape)
        return a.reshape(-1)[self.idx]

    def equals(self, got) -> bool:
        """np.array_equal of a full array with the reference output, at the stored positions."""
        return np.array_equal(self.take(got), self.values)

    def diff(self, got) -> np.ndarray:
        """got - reference at the stored positions."""
        return self.take(got) - self.values

    def nonfinite(self) -> int:
        """How many elements of the whole reference output are NaN or infinite (all of them are stored)."""
        return int((~np.isfinite(self.values)).sum())

    def same_nan(self, got) -> bool:
        """The NaN pattern of a full array equals the reference's (every non-finite reference element is stored)."""
        nan = np.isnan(self.values)
        return np.array_equal(np.isnan(self.take(got)), nan) and int(np.isnan(got).sum()) == int(nan.sum())

    def rows(self) -> np.ndarray:
        """Row (leading-axes flat) index of every stored element."""
        return self.idx // (self.shape[-1] if self.shape and self.shape[-1] else 1)

    def row_absmax_at(self) -> np.ndarray:
        """The largest finite magnitude of the row of every stored element (overall when there are many rows)."""
        return self.row_absmax[self.rows()] if self.row_absmax.size > 1 else np.full(self.idx.size, self.absmax())

    def absmax(self) -> float:
        return float(self.row_absmax.max()) if self.row_absmax.size else 0.0


class _Store:
    """tests/golden/reference_outputs.*: per test id a list of events; the sampled arrays are packed into three pools
    (sorted flat indices as deltas, values as float32, row maxima)."""

    def __init__(self):
        self.events, self.recorded = {}, {}
        if os.path.exists(JSON_PATH):
            with open(JSON_PATH) as f:
                self.events = json.load(f)
            pools = np.load(NPZ_PATH)
            self.idx_pool, self.val_pool, self.row_pool = pools["idx_delta"], pools["values"], pools["row_absmax"]

    def sample(self, ev) -> Sample:
        i0, n = ev["idx"]
        r0, nr = ev["rows"]
        dtype = np.dtype(ev["dtype"])
        width = 2 if dtype.kind == "c" else 1
        idx = np.cumsum(self.idx_pool[i0:i0 + n].astype(np.int64))
        values = self.val_pool[ev["values"]:ev["values"] + n * width].copy().view(dtype)
        return Sample(ev["shape"], dtype, idx, values, self.row_pool[r0:r0 + nr])

    def save(self):
        """Writes the recorded tests together with the stored ones that were not run again."""
        merged = {t: [dict(ev, _sample=self.sample(ev)) if "shape" in ev else ev for ev in evs]
                  for t, evs in self.events.items() if t not in self.recorded}
        merged.update(self.recorded)
        idx, vals, rows, out = [], [], [], {}
        at = [0, 0, 0]
        for test_id in sorted(merged):
            out[test_id] = []
            for ev in merged[test_id]:
                ev = dict(ev)
                s = ev.pop("_sample", None)
                if s is not None:
                    v = np.ascontiguousarray(s.values).view(np.float32)
                    ev.update(shape=list(s.shape), dtype=s.dtype.str, idx=[at[0], int(s.idx.size)], values=at[1],
                              rows=[at[2], int(s.row_absmax.size)])
                    idx.append(np.diff(s.idx, prepend=0))
                    vals.append(v)
                    rows.append(s.row_absmax.reshape(-1).astype(np.float32))
                    at = [at[0] + s.idx.size, at[1] + v.size, at[2] + s.row_absmax.size]
                out[test_id].append(ev)
        cat = lambda parts, dt: np.concatenate(parts).astype(dt) if parts else np.zeros(0, dt)
        np.savez_compressed(NPZ_PATH, idx_delta=cat(idx, np.uint32), values=cat(vals, np.float32),
                            row_absmax=cat(rows, np.float32))
        with open(JSON_PATH, "w") as f:
            json.dump(out, f, separators=(",", ":"), sort_keys=True)
            f.write("\n")


STORE = _Store()


class Reference:
    """oracle/ref.py's call surface for one test: replayed from the store, or run live and recorded."""

    def __init__(self, test_id: str):
        self.test_id = test_id
        self._pos = 0
        self._inputs = 0              # running crc32 of everything this test handed the reference
        self._warned = False
        if RECORD:
            from oracle import ref as live
            if not live.available():
                raise RuntimeError("B200_RECORD_REFERENCE needs oracle/_ref/libjst_ref.so (oracle/build_ref.sh)")
            self._live = live
            STORE.recorded[test_id] = []
        else:
            self._live = None
        self.RefError = RefError

    # -- one call: run + record, or replay -------------------------------------------------------------------------
    def _call(self, name, run, args=(), produces=True):
        self._inputs = _crc(_crc(self._inputs, name), args)
        if self._live is not None:
            events = STORE.recorded[self.test_id]
            try:
                out = run()
            except self._live.RefError as exc:
                events.append({"call": name, "error": str(exc), "in": self._inputs})
                raise RefError(str(exc)) from None
            if not produces:
                return out
            ev = {"call": name, "in": self._inputs}
            if isinstance(out, np.ndarray):
                ev["_sample"] = out = Sample.of(f"{self.test_id}#{len(events)}", out)
            else:
                ev["value"] = out
            events.append(ev)
            return out
        events = STORE.events.get(self.test_id)
        if events is None:
            raise KeyError(f"no stored reference outputs for {self.test_id}: record them with B200_RECORD_REFERENCE=1")
        ev = events[self._pos] if self._pos < len(events) else None
        if not produces and (ev is None or ev["call"] != name or "error" not in ev):
            return None                                 # calls without a result are recorded only when they failed
        if ev is None or ev["call"] != name:
            raise AssertionError(f"{self.test_id}: call {name} where the recording has {ev}: record it again")
        self._pos += 1
        if ev.get("in") != self._inputs and not self._warned:
            self._warned = True
            warnings.warn(f"{self.test_id}: the inputs handed to the reference differ from those its stored outputs were "
                          "recorded for; if the test fails, record them again (B200_RECORD_REFERENCE=1)")
        if "error" in ev:
            raise RefError(ev["error"])
        if "shape" in ev:
            return STORE.sample(ev)
        return ev["value"]

    # -- module-level one-shot wrappers of oracle/ref.py -----------------------------------------------------------
    def run_block(self, *a, **kw):
        return self._call("run_block", lambda: self._live.run_block(*a, **kw), (a, kw))

    def window(self, n):
        return self._call("window", lambda: self._live.window(n), (n,))

    def fft(self, *a, **kw):
        return self._call("fft", lambda: self._live.fft(*a, **kw), (a, kw))

    def multiply(self, a, b):
        return self._call("multiply", lambda: self._live.multiply(a, b), (a, b))

    def amplitude(self, *a, **kw):
        return self._call("amplitude", lambda: self._live.amplitude(*a, **kw), (a, kw))

    def range_(self, *a, **kw):
        return self._call("range_", lambda: self._live.range_(*a, **kw), (a, kw))

    def spectrum_engine(self, *a, **kw):
        return self._call("spectrum_engine", lambda: self._live.spectrum_engine(*a, **kw), (a, kw))

    def Session(self, log_level: int = 1):
        return _Session(self, log_level)

    def VizSession(self, *a, **kw):
        return _VizSession(self, *a, **kw)


class _Session:
    def __init__(self, ref: Reference, log_level: int):
        self._ref = ref
        self._s = ref._call("Session", lambda: ref._live.Session(log_level), (log_level,), produces=False)

    def __enter__(self):
        return self

    def __exit__(self, *a):
        if self._s is not None:
            self._s.close()

    def _void(self, name, *a, **kw):
        full = [v.full if isinstance(v, Sample) else v for v in a]     # a reference output fed to a later stage
        return self._ref._call("Session." + name, lambda: getattr(self._s, name)(*full, **kw), (a, kw), produces=False)

    def add_source(self, *a, **kw):
        self._void("add_source", *a, **kw)

    def write_source(self, *a, **kw):
        self._void("write_source", *a, **kw)

    def add_block(self, *a, **kw):
        self._void("add_block", *a, **kw)

    def reconfigure(self, *a, **kw):
        self._void("reconfigure", *a, **kw)

    def compute(self):
        self._void("compute")

    def output(self, block, port, select=None):
        """`select` (e.g. a decimating slice) is applied to the full output before it is sampled and stored."""
        return self._ref._call("Session.output", lambda: (select or (lambda a: a))(self._s.output(block, port)),
                              (block, port))

    def output_info(self, block, port):
        info = dict(self._ref._call("Session.output_info", lambda: _jsonable(self._s.output_info(block, port)),
                                           (block, port)))
        info["shape"] = tuple(info["shape"])
        return info


class _VizSession:
    def __init__(self, ref: Reference, *a, **kw):
        self._ref = ref
        self._v = ref._call("VizSession", lambda: ref._live.VizSession(*a, **kw), (a, kw), produces=False)

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def close(self):
        if self._v is not None:
            self._v.close()

    def compute(self, x):
        full = x.full if isinstance(x, Sample) else x
        self._ref._call("VizSession.compute", lambda: self._v.compute(full), (x,), produces=False)

    def reconfigure(self, config):
        self._ref._call("VizSession.reconfigure", lambda: self._v.reconfigure(config), (config,), produces=False)

    def read(self, select=None):
        """`select` (e.g. a reshape) is applied to the full output before it is sampled and stored."""
        return self._ref._call("VizSession.read", lambda: (select or (lambda a: a))(self._v.read()))

    def write_index(self):
        return self._ref._call("VizSession.write_index", lambda: self._v.write_index())


def _jsonable(info: dict) -> dict:
    return {k: (list(v) if isinstance(v, tuple) else (np.dtype(v).str if k == "dtype" and v is not None else v))
            for k, v in info.items()}
