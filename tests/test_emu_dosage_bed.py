"""test_gpu_dosage_bed.py under the warp emulator (see test_emu_resident.py): the same .bed-mode cases, with the product's
kernel and C-ABI sources compiled with g++ and "device" buffers in host memory."""
import functools
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))
import test_gpu_dosage_bed as D
import test_gpu_resident as R
from test_emu_resident import _clone, emu_api  # noqa: F401  (emu_api is a fixture)


@pytest.fixture
def mem():
    return R.HostMem()


@pytest.fixture
def resident(mem):
    return functools.partial(R.run_resident, mem)


# the 4.4 GB launch and the torch wrapper over device tensors stay on the GPU
_SKIP = {"test_bed_rows_past_4_gib", "test_bed_torch_wrapper_device"}
for _name, _fn in sorted(vars(D).items()):
    if _name.startswith("test_") and callable(_fn) and _name not in _SKIP:
        globals()[_name + "_emulated"] = _clone(_fn)
