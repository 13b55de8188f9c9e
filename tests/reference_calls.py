"""The original Octopus code's answers, recorded once and replayed by the tests that compare against it.

Those tests call the original code through the ctypes wrappers of oracle/oracle.py (``RefKernel``, ``RefHMM``,
``RefErrorModel``), whose libraries are compiled from the Octopus sources (oracle/Makefile) and so exist only where those sources
are. The answers they gave on each test's seeded inputs are stored in tests/golden/reference_calls.json.xz and the fixtures
replay them in call order. One digest of all the calls' arguments is stored beside them; after the test, the replay checks
that the test made as many calls with the same arguments, so a test whose inputs change fails instead of passing against
stale answers. Answers that the tests only compare for equality and that would be large (the error models' arrays) are
stored as a ``Digest``, which compares equal to a value holding the same bytes.

Recording: build oracle/_ref (``make -C oracle REF=<Octopus source tree>``) and run the tests with
``PHMM_RECORD_REFERENCE=<output path>``. Every test that runs replaces its own entry; the others are kept from the committed
file. The GPU tests record on a GPU host.
"""
import atexit
import functools
import hashlib
import json
import lzma
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.json.xz")
RECORD = os.environ.get("PHMM_RECORD_REFERENCE")


def _feed(h, x):
    if isinstance(x, np.generic):
        x = x.item()
    if isinstance(x, np.ndarray):                      # shape and bytes: an int8 and a uint8 view of one array hash alike
        h.update(b"A%r" % (x.shape,))
        h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, (bytes, bytearray, str)):
        b = x.encode() if isinstance(x, str) else bytes(x)
        h.update(b"B%d:" % len(b))
        h.update(b)
    elif isinstance(x, (list, tuple)):
        h.update(b"L%d" % len(x))
        for e in x:
            _feed(h, e)
    elif isinstance(x, dict):
        h.update(b"D%d" % len(x))
        for k in sorted(x):
            _feed(h, k)
            _feed(h, x[k])
    elif hasattr(x, "arrays"):                          # HaplotypeBlock / ReadBlock
        _feed(h, x.arrays())
    else:
        h.update(b"V%s:%r" % (type(x).__name__.encode(), x))


class Digest:
    """A recorded answer kept as a 32-bit hash: equal to any value with the same shapes and bytes."""

    def __init__(self, hexdigest):
        self.hex = hexdigest

    @classmethod
    def of(cls, value):
        h = hashlib.blake2b(digest_size=4)
        _feed(h, value)
        return cls(h.hexdigest())

    def __eq__(self, other):
        return self.hex == (other if isinstance(other, Digest) else Digest.of(other)).hex

    def __repr__(self):
        return "Digest(%s)" % self.hex


# answers stored as digests: what the test sees in place of the original's return value, in both modes
_DIGESTED = {
    "errmodel.tandem_repeats": Digest.of,
    "errmodel.reset": lambda r: (r["rc"], Digest.of({k: v for k, v in r.items() if k != "rc"})),
}


def _enc(v):
    if isinstance(v, Digest):
        return {"h": v.hex}
    if isinstance(v, np.ndarray):
        return {"a": v.dtype.str, "s": list(v.shape), "v": v.ravel().tolist()}
    if isinstance(v, tuple):
        return {"t": [_enc(x) for x in v]}
    if isinstance(v, list):
        return [_enc(x) for x in v]
    return v.item() if isinstance(v, np.generic) else v


def _dec(v):
    if isinstance(v, list):
        return [_dec(x) for x in v]
    if isinstance(v, dict):
        if "h" in v:
            return Digest(v["h"])
        if "a" in v:
            return np.asarray(v["v"], dtype=np.dtype(v["a"])).reshape(v["s"])
        return tuple(_dec(x) for x in v["t"])
    return v


@functools.lru_cache(maxsize=None)
def _load():
    if not os.path.exists(GOLDEN):
        return {"tests": {}}
    with lzma.open(GOLDEN, "rt") as f:
        return json.load(f)


_recorded = {}


def _save():
    old = _load()
    tests = dict(old["tests"])
    tests.update({k: {"calls": s["calls"], "args": s["args"].hexdigest(), "isas": s["isas"]} for k, s in _recorded.items()})
    with lzma.open(RECORD, "wt", preset=9 | lzma.PRESET_EXTREME) as f:
        json.dump({"tests": tests}, f, sort_keys=True, separators=(",", ":"))


class _Proxy:
    """One of the original's objects as a test sees it: calls go to ``state['call']`` under ``prefix + method``."""

    def __init__(self, state, prefix):
        self._state, self._prefix = state, prefix

    def __getattr__(self, method):
        def call(*args, **kwargs):
            name = self._prefix + method
            _feed(self._state["args"], [name, list(args), kwargs])
            return self._state["call"](name, args, kwargs)
        return call


def _record_state(key, live, isas):
    state = {"calls": [], "args": hashlib.blake2b(digest_size=8), "isas": isas}

    def call(name, args, kwargs):
        obj, method = name.split(".")
        result = getattr(live[obj], method)(*args, **kwargs)
        result = _DIGESTED.get(name, lambda r: r)(result)
        state["calls"].append([name, _enc(result)])
        return result
    state["call"] = call
    if not _recorded:
        atexit.register(_save)
    _recorded[key] = state
    return state


def _replay_state(key, rec):
    state = {"i": 0, "args": hashlib.blake2b(digest_size=8), "isas": rec["isas"]}

    def call(name, args, kwargs):
        i = state["i"]
        assert i < len(rec["calls"]), "%s: call %d to the original code, only %d recorded" % (key, i + 1, len(rec["calls"]))
        assert rec["calls"][i][0] == name, "%s: call %d is %s, recorded %s" % (key, i + 1, name, rec["calls"][i][0])
        state["i"] = i + 1
        return _dec(rec["calls"][i][1])

    def check():
        assert state["i"] == len(rec["calls"]), "%s: %d calls to the original code, %d recorded" % (key, state["i"], len(rec["calls"]))
        assert state["args"].hexdigest() == rec["args"], "%s: the calls' arguments differ from the recorded ones: re-record" % key
    state["call"], state["check"] = call, check
    return state


def reference(request, what):
    """The original code behind a fixture: 'kernels' ({isa: RefKernel}), 'hmm' (RefHMM) or 'errmodel' (RefErrorModel).
    Replayed from GOLDEN, or with PHMM_RECORD_REFERENCE set, called live and recorded."""
    key = request.node.nodeid.split("/")[-1]
    state = request.node.__dict__.get("_reference_calls")
    if state is None:
        if RECORD:
            from oracle.oracle import RefErrorModel, RefHMM, RefKernel, available_ref_isas
            assert available_ref_isas() and RefHMM.available() and RefErrorModel.available(), "recording needs every oracle/_ref library"
            live = {isa: RefKernel(isa) for isa in available_ref_isas()}
            live.update(hmm=RefHMM(), errmodel=RefErrorModel())
            state = _record_state(key, live, available_ref_isas())
        else:
            rec = _load()["tests"].get(key)
            if rec is None:
                pytest.fail("no recorded answers of the original code for %s in %s" % (key, GOLDEN))
            state = _replay_state(key, rec)
            request.addfinalizer(state["check"])
        request.node._reference_calls = state
    if what == "kernels":
        return {isa: _Proxy(state, isa + ".") for isa in state["isas"]}
    return _Proxy(state, what + ".")
