"""Calls into the original OV²SLAM code, replayed from stored results.

The tests named test_oracle_vs_reference_* compare the oracle with functions of the original project compiled from its own
sources (the recipes under oracle/ref_build/, into oracle/_ref/).  Those sources are not part of this repository, so what each
such call wrote is stored under tests/golden/ref_<module>.npz and the tests compare against the stored results: `library()`
stands in for the ctypes library, checks that each call gets the inputs it was recorded with and writes back into the caller's
arrays what the original code wrote there.

With OV2SLAM_RECORD=1 and the original sources at hand (the recipes compile them), the same tests call the real libraries and
rewrite the golden files:  OV2SLAM_RECORD=1 python -m pytest tests/test_oracle_vs_reference_*.py
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
from pathlib import Path

import numpy as np
import pytest

GOLDEN = Path(__file__).resolve().parent / "golden"
RECORD = os.environ.get("OV2SLAM_RECORD") == "1"
_SCALARS = (C.c_int, C.c_int32, C.c_uint8, C.c_float, C.c_double)


def _test_name() -> str:
    # "tests/test_x.py::test_y[params] (call)" -> "test_y[params]"
    return os.environ["PYTEST_CURRENT_TEST"].split("::", 1)[1].rsplit(" ", 1)[0]


def _array(arg):
    """The numpy array behind a `ndarray.ctypes.data_as(...)` pointer (numpy keeps it on the pointer), else None."""
    arr = getattr(arg, "_arr", None)
    return arr if isinstance(arr, np.ndarray) else None


def _byref(arg):
    """The ctypes scalar behind `ctypes.byref(x)`, else None."""
    obj = getattr(arg, "_obj", None)
    return obj if isinstance(obj, _SCALARS) else None


def _input_summary(arg):
    """What identifies an input: size, sum and sum of magnitudes of an array; the value of a scalar; None for handles."""
    a = _array(arg)
    if a is not None:
        v = a.astype(np.float64).ravel()
        return np.array([v.size, v.sum(), np.abs(v).sum()])
    s = _byref(arg)
    if s is not None:
        return np.array([float(s.value)])
    if isinstance(arg, _SCALARS):
        return np.array([float(arg.value)])
    if isinstance(arg, (bool, int, float, np.integer, np.floating)):
        return np.array([float(arg)])
    return None


def _same_input(got, want) -> bool:
    if got.shape != want.shape or (len(got) == 3 and got[0] != want[0]):
        return False
    scale = got[-1] if len(got) == 3 else abs(want[0])
    # stored as float32; a last-bit difference of numpy's BLAS on another machine must not matter either
    return bool(np.all(np.abs(got - want) <= 1e-6 * max(scale, 1.0)))


class _Recorder:
    """The real library; every call's outputs (arrays and byref scalars it changed, the return value) are kept for save()."""

    def __init__(self, lib):
        self._lib, self._calls = lib, {}

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*args):
            before = [None if _array(a) is None else _array(a).copy() for a in args]
            summ = [_input_summary(a) for a in args]
            ret = fn(*args)
            ins = {i: s for i, s in enumerate(summ) if s is not None}
            outs = {}
            for i, a in enumerate(args):
                arr, s = _array(a), _byref(a)
                if arr is not None and not np.array_equal(arr, before[i]):
                    outs[i] = arr.copy()
                elif s is not None:
                    outs[i] = np.array(s.value)
            self._calls.setdefault(_test_name(), []).append((name, np.nan if ret is None else ret, ins, outs))
            return ret

        return _Fn(call, fn)

    def save(self, path: Path):
        # per test: the call names, the return values, and per dtype one vector of all input summaries (float32) or outputs
        # (their own dtype) with a (call, argument, size) index
        flat = {}
        for t, calls in self._calls.items():
            flat[f"{t}|fn"] = np.array([c[0] for c in calls])
            flat[f"{t}|ret"] = np.array([c[1] for c in calls], np.float64)
            for j, kind in ((2, "in"), (3, "out")):
                groups = {}
                for k, c in enumerate(calls):
                    for i, v in c[j].items():
                        v = np.asarray(v, np.float32 if kind == "in" else None).ravel()
                        at, data = groups.setdefault(v.dtype.name, ([], []))
                        at.append((k, i, v.size))
                        data.append(v)
                for dt, (at, data) in groups.items():
                    flat[f"{t}|{kind}.{dt}"] = np.concatenate(data)
                    flat[f"{t}|{kind}.{dt}_at"] = np.array(at, np.int32)
        np.savez_compressed(path, **flat)


class _Replay:
    """Answers each call with the recorded outputs of the same call (same test, same position, same inputs)."""

    def __init__(self, path: Path):
        self._calls, self._next = {}, {}
        with np.load(path) as z:
            for t in {key.rsplit("|", 1)[0] for key in z.files}:
                calls = [dict(fn=str(f), ret=r, ins={}, outs={}) for f, r in zip(z[f"{t}|fn"], z[f"{t}|ret"])]
                for key in z.files:
                    if key.startswith(t + "|") and key.endswith("_at"):
                        data, kind, at = z[key[:-3]], key[len(t) + 1:].split(".")[0], z[key]
                        ends = np.cumsum(at[:, 2])
                        for (k, i, n), b in zip(at, ends):
                            calls[k][kind + "s"][int(i)] = data[b - n:b]
                self._calls[t] = calls

    def __getattr__(self, name):
        def call(*args):
            t = _test_name()
            k = self._next.get(t, 0)
            self._next[t] = k + 1
            calls = self._calls.get(t, [])
            assert k < len(calls), f"{t}: no recorded call #{k} ({name}) of the original code"
            rec = calls[k]
            assert rec["fn"] == name, f"{t}: call #{k} is {name}, the recording has {rec['fn']}"
            for i, a in enumerate(args):
                s = _input_summary(a)
                if s is not None and i in rec["ins"]:
                    assert _same_input(s, rec["ins"][i]), f"{t}: argument {i} of {name} (call #{k}) is not the recorded input"
                if i in rec["outs"]:
                    arr, obj = _array(a), _byref(a)
                    if arr is not None:
                        arr[...] = rec["outs"][i].reshape(arr.shape)
                    else:
                        obj.value = type(obj.value)(rec["outs"][i][0])
            ret = float(rec["ret"])
            return None if np.isnan(ret) else int(ret) if ret == int(ret) else ret

        return _Fn(call, None)


class _Fn:
    """A library function; attribute writes (restype, argtypes) go to the real function when there is one."""

    def __init__(self, call, real):
        object.__setattr__(self, "_call", call)
        object.__setattr__(self, "_real", real)

    def __call__(self, *args):
        return self._call(*args)

    def __setattr__(self, key, value):
        if self._real is not None:
            setattr(self._real, key, value)


@contextlib.contextmanager
def library(module: str, load):
    """The original code's library for the tests of `module`: replayed from tests/golden/ref_<module>.npz, or with
    OV2SLAM_RECORD=1 the real one, `load()` (None when it cannot be built), whose calls then rewrite that file."""
    path = GOLDEN / f"ref_{module}.npz"
    if not RECORD:
        yield _Replay(path)
        return
    lib = load()
    if lib is None:
        pytest.fail("OV2SLAM_RECORD=1 needs the original sources to build oracle/_ref/")
    rec = _Recorder(lib)
    yield rec
    rec.save(path)
