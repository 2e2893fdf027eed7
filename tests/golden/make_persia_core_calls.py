"""Records what the reference's own Python package (`persia`, PersiaML/PERSIA) asks of `persia_core` into
tests/golden/persia_core_calls.json, with this repository's persia_core installed in place of the Rust extension.

    python tests/golden/make_persia_core_calls.py <path to a PERSIA checkout>

Two scenarios are recorded, each from a fresh import of `persia`:
  * package_surface      — the reference's data / optim / embedding-config classes driven the way its test suite does;
  * reference_test_data  — the reference's test/embedding/test_data.py, run by pytest as it stands.
Every name the package reads from a persia_core module and every call it makes (arguments, and the type of the result or
of the exception) is stored; tests/test_persia_core_surface.py replays them, so the surface stays checked against what
the reference package uses without the reference tree.  Only the call trace is stored, none of the package's code."""
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "persia_core_calls.json")


class Recorder:
    def __init__(self):
        self.events, self.handles, self.seen = [], 0, set()

    def enc(self, v):
        if isinstance(v, Obj):
            return {"handle": v._h}
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        if isinstance(v, bytes):
            return {"bytes": v.hex()}
        if isinstance(v, np.ndarray):
            return {"ndarray": {"dtype": v.dtype.str, "shape": list(v.shape), "data": v.reshape(-1).tolist()}}
        if isinstance(v, np.dtype):
            return {"dtype": v.str}
        if isinstance(v, type) and issubclass(v, np.generic):
            return {"nptype": np.dtype(v).str}
        if isinstance(v, np.generic):
            return {"npscalar": {"dtype": v.dtype.str, "value": v.item()}}
        if isinstance(v, (list, tuple)):
            return {type(v).__name__: [self.enc(x) for x in v]}
        raise TypeError(f"cannot record an argument of type {type(v)}")

    def wrap(self, target, fn):
        def call(*args, **kwargs):
            ev = {"op": "call", "target": target, "args": [self.enc(a) for a in args],
                  "kwargs": {k: self.enc(v) for k, v in kwargs.items()}}
            self.events.append(ev)
            try:
                r = fn(*[unwrap(a) for a in args], **{k: unwrap(v) for k, v in kwargs.items()})
            except Exception as e:
                ev["result"] = {"raises": type(e).__name__}
                raise
            if type(r).__module__ == "persia_b200.persia_core":
                self.handles += 1
                ev["result"] = {"handle": self.handles}
                return Obj(self, self.handles, r)
            ev["result"] = {"type": type(r).__name__}
            return r

        return call

    def module(self, real, name):
        rec = self

        class RecModule(types.ModuleType):
            def __getattribute__(self, attr):
                v = super().__getattribute__(attr)
                # prelude.register_submodule walks dir(module) and keeps the submodules only: the names it merely
                # looks at are not part of what the package needs
                if (not attr.startswith("_") and (isinstance(v, types.ModuleType) or
                                                  sys._getframe(1).f_code.co_name != "register_submodule")
                        and (name, attr) not in rec.seen):
                    rec.seen.add((name, attr))
                    rec.events.append({"op": "getattr", "target": f"{name}.{attr}"})
                return v

        m = RecModule(name)
        for k in dir(real):
            if k.startswith("__"):
                continue
            v = getattr(real, k)
            if isinstance(v, types.ModuleType):
                v = self.module(v, f"{name}.{k}")
            elif callable(v):
                v = self.wrap(f"{name}.{k}", v)
            setattr(m, k, v)
        return m


class Obj:
    """An object persia_core returned: its method calls are recorded against the handle it was given."""

    def __init__(self, rec, h, real):
        object.__setattr__(self, "_rec", rec)
        object.__setattr__(self, "_h", h)
        object.__setattr__(self, "_real", real)

    def __getattr__(self, name):
        v = getattr(self._real, name)
        if callable(v):
            return self._rec.wrap(f"${self._h}.{name}", v)
        self._rec.events.append({"op": "getattr", "target": f"${self._h}.{name}", "type": type(v).__name__})
        return v


def unwrap(v):
    if isinstance(v, Obj):
        return v._real
    if isinstance(v, (list, tuple)):
        return type(v)(unwrap(x) for x in v)
    return v


def fresh(ref):
    """A recorder installed as persia_core, and no `persia` module imported yet."""
    from persia_b200 import persia_core

    persia_core.reset()
    facade = persia_core.install()
    rec = Recorder()
    root = rec.module(facade, "persia_core")
    sys.modules["persia_core"] = root
    for n in ("data", "forward", "backward", "optim", "utils", "nats"):
        sys.modules[f"persia_core.{n}"] = getattr(root, n)
    for k in [k for k in sys.modules if k == "persia" or k.startswith("persia.")]:
        del sys.modules[k]
    if ref not in sys.path:
        sys.path.insert(0, ref)
    return rec


def package_surface():
    import persia  # noqa: F401
    from persia.embedding import EmbeddingConfig
    from persia.embedding.data import IDTypeFeature, IDTypeFeatureWithSingleID, Label, NonIDTypeFeature, PersiaBatch
    from persia.embedding.optim import SGD, Adagrad, Adam

    batch_size = 5
    for dt in (np.bool_, np.int8, np.int16, np.int32, np.int64, np.float32, np.float64, np.uint8):
        NonIDTypeFeature(np.zeros((batch_size, 3), dtype=dt))
    ids = [IDTypeFeature("f1", [np.array([1, 2], np.uint64) for _ in range(batch_size)]),
           IDTypeFeatureWithSingleID("f2", np.arange(batch_size, dtype=np.uint64))]
    try:
        PersiaBatch(ids, requires_grad=True)
    except Exception:
        pass
    else:
        raise AssertionError("requires_grad without labels was accepted")
    pb = PersiaBatch(ids, non_id_type_features=[NonIDTypeFeature(np.ones((batch_size, 2), np.float32))],
                     labels=[Label(np.ones((batch_size, 1), np.float32))], requires_grad=True, meta=b"m")
    assert isinstance(pb.to_bytes(), bytes)
    SGD(0.1).optimizer_base, Adagrad(0.1).optimizer_base, Adam(1e-3).optimizer_base  # noqa: B018
    cfg = EmbeddingConfig()
    assert cfg.weight_bound == 10 and cfg.admit_probability == 1.0


def reference_test_data(ref):
    import pytest

    path = os.path.join(ref, "test", "embedding", "test_data.py")
    rc = pytest.main(["-q", "-p", "no:cacheprovider", "--rootdir", os.path.dirname(path), path])
    assert rc == 0, rc


def main():
    ref = os.path.abspath(sys.argv[1])
    sys.path.insert(0, ROOT)
    sys.dont_write_bytecode = True
    try:
        import colorlog  # noqa: F401
    except ImportError:  # the reference's logger wants colorlog; give it a plain formatter
        import logging

        m = types.ModuleType("colorlog")
        m.ColoredFormatter = lambda fmt=None, *a, **k: logging.Formatter("%(levelname)s %(message)s")
        sys.modules["colorlog"] = m
    out = {"source": "persia/ (Python package) and test/embedding/test_data.py of PersiaML/PERSIA",
           "scenarios": {}}
    rec = fresh(ref)
    package_surface()
    out["scenarios"]["package_surface"] = rec.events
    rec = fresh(ref)
    reference_test_data(ref)
    out["scenarios"]["reference_test_data"] = rec.events
    with open(DST, "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")
    print(DST, {k: len(v) for k, v in out["scenarios"].items()})


if __name__ == "__main__":
    main()
