"""The host side of the five tools without a GPU: the real executables' sources (vcfx_b200/tools) linked against the
emulator build of the library (tests/emu/), run through the cases of tests/test_gpu_cli.py against the reference
tools (tests/reference_runs.py: the reference build where there is one, else recorded outputs) — with one context and
with several contexts in one process (VCFX_CUDA_DEVICES: chunks dealt round-robin over the devices, text written in
submission order)."""
import inspect
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))
import test_gpu_cli as G


@pytest.fixture(scope="module")
def emu_bin():
    import build_emu
    return build_emu.build_tools()


@pytest.fixture(params=["0", "0,1,2"], ids=["one-device", "three-devices"])
def emu_env(request, emu_bin, monkeypatch):
    monkeypatch.setattr(G, "BIN", emu_bin)
    monkeypatch.setenv("VCFX_EMU_DEVICES", "3")
    monkeypatch.setenv("VCFX_CUDA_DEVICES", request.param)
    return request.param


files = G.files          # the module-scoped input files of the GPU CLI tests


def _clone(fn):
    sig = inspect.signature(fn)
    params = list(sig.parameters.values()) + [inspect.Parameter("emu_env", inspect.Parameter.POSITIONAL_OR_KEYWORD)]

    def w(**kw):
        kw.pop("emu_env")
        return fn(**kw)
    w.__signature__ = sig.replace(parameters=params)
    w.__name__ = fn.__name__ + "_emulated"
    w.__doc__ = fn.__doc__
    marks = [m for m in getattr(fn, "pytestmark", []) if m.name != "gpu"]
    if marks:
        w.pytestmark = marks
    return w


# (files of tens of MB and the multi-GPU hardware test stay on the GPU)
_SKIP = {"test_large_file_parallel_io", "test_multi_gpu_same_bytes"}
for _name, _fn in sorted(vars(G).items()):
    if _name.startswith("test_") and callable(_fn) and _name not in _SKIP:
        globals()[_name + "_emulated"] = _clone(_fn)
