"""test_gpu_king.py under the warp emulator (see test_emu_resident.py): the product's kernel and C-ABI sources compiled
with g++, "device" memory in host memory, and tcgen05.mma emulated from the shared-memory and instruction descriptors it
is given, so a wrong descriptor or planes layout fails here.  The emulator's planes hold 1 MiB, so slab borders fall at a
few hundred rows; 2,504 samples, the pedigree, the C2 shape and the torch device paths stay on the GPU."""
import functools
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))
import test_gpu_king as K
import test_gpu_resident as R
from test_emu_resident import _clone, emu_api  # noqa: F401  (emu_api is a fixture)


@pytest.fixture
def resident():
    return functools.partial(R.run_resident, R.HostMem())


_SKIP = {"test_king_end_to_end_and_device_bed", "test_king_simulated_pedigree", "test_king_c2_shape_against_matmul"}
for _name, _fn in sorted(vars(K).items()):
    if _name.startswith("test_") and callable(_fn) and _name not in _SKIP:
        globals()[_name + "_emulated"] = _clone(_fn)
