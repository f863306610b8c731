"""test_gpu_resident.py under the warp emulator (see test_emu_parity.py): the same device-resident cases, with the
product's kernel and C-ABI sources compiled with g++ and "device" buffers in host memory."""
import functools
import inspect
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))
import test_gpu_resident as R


@pytest.fixture(scope="module")
def emu_api():
    import build_emu
    return build_emu.load_api()


@pytest.fixture
def mem():
    return R.HostMem()


@pytest.fixture
def resident(mem):
    return functools.partial(R.run_resident, mem)


def _clone(fn):
    sig = inspect.signature(fn)
    params = [p.replace(name="emu_api") if p.name == "cuda_api" else p for p in sig.parameters.values()]

    def w(**kw):
        kw["cuda_api"] = kw.pop("emu_api")
        return fn(**kw)
    w.__signature__ = sig.replace(parameters=params)
    w.__name__ = fn.__name__ + "_emulated"
    w.__doc__ = fn.__doc__
    marks = [m for m in getattr(fn, "pytestmark", []) if m.name != "gpu"]
    if marks:
        w.pytestmark = marks
    return w


# more than 2^20 dropped lines and the launch past 4 GiB stay on the GPU
_SKIP = {"test_resident_phase_checker_event_list_grows", "test_resident_one_launch_past_4_gib"}
for _name, _fn in sorted(vars(R).items()):
    if _name.startswith("test_") and callable(_fn) and _name not in _SKIP:
        globals()[_name + "_emulated"] = _clone(_fn)
