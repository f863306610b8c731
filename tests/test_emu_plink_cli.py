"""test_gpu_plink_cli.py without a GPU: VCFX_plink_bed's source linked against the emulator build of the library
(tests/emu/), with one context and with three contexts in one process (VCFX_CUDA_DEVICES: chunks dealt round-robin
over the devices, the .bed written in submission order)."""
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))
import test_gpu_plink_cli as P
from test_emu_cli import _clone


@pytest.fixture(scope="module")
def emu_bin():
    import build_emu
    return build_emu.build_tools()


@pytest.fixture(params=["0", "0,1,2"], ids=["one-device", "three-devices"])
def emu_env(request, emu_bin, monkeypatch):
    monkeypatch.setattr(P, "BIN", emu_bin)
    monkeypatch.setenv("VCFX_EMU_DEVICES", "3")
    monkeypatch.setenv("VCFX_CUDA_DEVICES", request.param)
    return request.param


files = P.files          # the module-scoped input files of the GPU tests

# (the hardware multi-GPU test stays on the GPU: the three-devices parameter covers the same dealing here)
_SKIP = {"test_multi_gpu_same_bytes"}
for _name, _fn in sorted(vars(P).items()):
    if _name.startswith("test_") and callable(_fn) and _name not in _SKIP:
        globals()[_name + "_emulated"] = _clone(_fn)
