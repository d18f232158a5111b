"""CPU: the stepped online controller's public record and the refusals of math_mpc_batch(actuator=...), without a CUDA
device.  The record mpcb_held_ctrl is part of the C ABI: its layout as g++ lays it out from include/mpcb200.h must be the
ctypes mirror _native.HeldCtrl, field for field."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_record_layout_matches_the_ctypes_mirror(tmp_path):
    from diplomjourney_b200 import _native
    exe = tmp_path / "held_ctrl_layout"
    r = subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "native", "held_ctrl_layout.cpp"), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    got = {ln.split()[0]: [int(x) for x in ln.split()[1:]] for ln in out if ln.strip()}
    R = _native.HeldCtrl
    assert got.pop("sizeof") == [ctypes.sizeof(R)] == [336]
    assert got.pop("alignof") == [ctypes.alignment(R)] == [8]
    assert got.pop("MPCB_LOOP_RUNNING") == [_native.LOOP_RUNNING, 0]
    assert list(got) == [name for name, _ in R._fields_]
    for name, (offset, size) in got.items():
        f = getattr(R, name)
        assert (f.offset, f.size) == (offset, size), name


@pytest.fixture
def mt():
    import importlib
    m = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    m._backend = None
    yield m
    m._backend = None


@pytest.mark.parametrize("extra, match", [
    (dict(isActual=False), "isActual=True"),
    (dict(rngs=[np.random.RandomState(1)]), "rngs"),
    (dict(seeds=[1]), "seeds"),
    (dict(device_noise=True), "device_noise"),
    (dict(host_loop=True), "host_loop"),
    (dict(logs=True), "logs"),
    (dict(rngs=[np.random.RandomState(1)], device_noise=True, logs=True), "rngs, device_noise, logs"),
])
def test_actuator_refusals_touch_no_solver_and_no_torch(mt, monkeypatch, extra, match):
    """Every combination the stepped run does not take is a ValueError raised before a solver (or torch) is touched:
    here no solver can be made at all, and importing torch would fail."""
    import builtins
    real_import = builtins.__import__

    def no_torch(name, *a, **k):
        if name == "torch" or name.startswith("torch."):
            raise AssertionError("torch imported")
        return real_import(name, *a, **k)

    def no_solver():
        raise AssertionError("solver touched")

    monkeypatch.setattr(builtins, "__import__", no_torch)
    monkeypatch.setattr(mt, "_solver", no_solver)
    kw = dict(isActual=True)
    kw.update(extra)
    with pytest.raises(ValueError, match=match):
        mt.math_mpc_batch([[0, 0, 0, 0, 0]], [[2, 3]], actuator=lambda c, r: c, **kw)


def test_actuator_must_be_callable(mt, monkeypatch):
    monkeypatch.setattr(mt, "_solver", lambda: (_ for _ in ()).throw(AssertionError("solver touched")))
    with pytest.raises(TypeError, match="callable"):
        mt.math_mpc_batch([[0, 0, 0, 0, 0]], [[2, 3]], isActual=True, actuator=42)
