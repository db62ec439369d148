"""Calls into the reference's compiled code that also run where it is not built.

A test reaches the reference through a `Reference`.  Where the compiled modules are present every call goes to them;
with SDET_RECORD_REFERENCE=1 in the environment (tests/golden/make_golden_reference_calls.py) the arguments and
results of each call are also written to tests/golden/reference_calls.json.  Where they are absent, the n-th call a
test makes is answered from that file: it must carry the arguments that were recorded, and every array it returns
is a `Recorded` stand-in (shape, dtype and a sha256 of the bytes the reference returned).  `same(ref, want)` compares
a reference result with an array bit for bit either way, so the tests keep their comparisons in both places."""
from __future__ import annotations

import atexit
import builtins
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.json")
RECORD = os.environ.get("SDET_RECORD_REFERENCE") == "1"
_recording: dict = {}
_replay = None
_count: dict = {}


def digest(a) -> str:
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)  # -0.0 -> +0.0: np.array_equal does not tell them apart either
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:32]


class Recorded:
    """What the reference returned for one array: enough to compare against, not the values."""

    def __init__(self, shape, dtype, sha):
        self.shape, self.dtype, self.sha = tuple(shape), np.dtype(dtype), sha

    @property
    def ndim(self):
        return len(self.shape)


def same(ref, want) -> bool:
    """ref (a reference result: an array, or its Recorded digest) equals `want` element for element."""
    w = np.asarray(want)
    if isinstance(ref, Recorded):
        if w.shape != ref.shape:
            return False
        wc = w.astype(ref.dtype)
        return bool(np.array_equal(wc, w)) and digest(wc) == ref.sha
    r = np.asarray(ref)
    ok = bool(np.array_equal(r, w))
    if ok and RECORD and isinstance(ref, np.ndarray):  # the digest comparison must agree with the one made here
        assert digest(w.astype(r.dtype)) == digest(r), "array_equal and the digest comparison disagree"
    return ok


def _arg(x) -> str:
    if isinstance(x, Recorded):
        return "a" + x.sha
    if isinstance(x, np.ndarray):
        return "a" + digest(x)
    if isinstance(x, (list, tuple)):
        return "[" + ",".join(_arg(v) for v in x) + "]"
    if isinstance(x, dict):
        return "{" + ",".join(f"{k}:{_arg(v)}" for k, v in sorted(x.items())) + "}"
    if isinstance(x, np.generic):
        return repr(x.item()) + x.dtype.str
    return repr(x)


def _enc(x):
    if isinstance(x, np.ndarray):
        return {"array": [list(x.shape), x.dtype.str, digest(x)]}
    if isinstance(x, tuple):
        return {"tuple": [_enc(v) for v in x]}
    if isinstance(x, list):
        return [_enc(v) for v in x]
    if isinstance(x, np.generic):
        return x.item()
    assert x is None or isinstance(x, (bool, int, float, str)), type(x)
    return x


def _dec(x):
    if isinstance(x, dict):
        return Recorded(*x["array"]) if "array" in x else tuple(_dec(v) for v in x["tuple"])
    if isinstance(x, list):
        return [_dec(v) for v in x]
    return x


def _test_id() -> str:
    cur = os.environ["PYTEST_CURRENT_TEST"].rsplit(" ", 1)[0]
    return cur.rsplit("/", 1)[-1]  # "test_module.py::test_name[params]", wherever pytest was started


def _save():
    rec = json.load(open(PATH)) if os.path.exists(PATH) else {}
    rec.update(_recording)
    with open(PATH, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(rec[k], separators=(',', ':'))}"
                                   for k in sorted(rec)) + "\n}\n")


class Reference:
    """`Reference(target)` forwards `ref.fn(*args, **kw)` to `target.fn`; `Reference(None)` replays the recording."""

    def __init__(self, target):
        self.live = target is not None
        self._target = target
        if RECORD and not self.live:
            raise RuntimeError("SDET_RECORD_REFERENCE=1 needs the compiled reference")

    def __getattr__(self, fn):
        return lambda *a, **k: self._call(fn, a, k)

    def _call(self, fn, args, kwargs):
        tid = _test_id()
        i = _count[tid] = _count.get(tid, -1) + 1
        key = hashlib.sha256(_arg([args, kwargs]).encode()).hexdigest()[:16]
        if self.live:
            try:
                res = getattr(self._target, fn)(*args, **kwargs)
                out = _enc(res)
            except Exception as e:
                out = {"raises": [type(e).__name__, str(e)]}
                if RECORD:
                    _recording.setdefault(tid, []).append([fn, key, out])
                raise
            if RECORD:
                _recording.setdefault(tid, []).append([fn, key, out])
            return res
        global _replay
        if _replay is None:
            _replay = json.load(open(PATH))
        calls = _replay.get(tid)
        assert calls is not None and i < len(calls), f"{tid}: no recorded reference call #{i}"
        rfn, rkey, out = calls[i]
        assert (rfn, rkey) == (fn, key), (f"{tid}: call #{i} {fn}() is not the call that was recorded; re-record with "
                                          "tests/golden/make_golden_reference_calls.py")
        if isinstance(out, dict) and "raises" in out:
            raise getattr(builtins, out["raises"][0], RuntimeError)(out["raises"][1])
        return _dec(out)


if RECORD:
    atexit.register(_save)
