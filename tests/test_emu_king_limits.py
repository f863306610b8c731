"""test_gpu_king_limits.py's refusals under the warp emulator (see test_emu_king.py): sample counts past the tile word
and past uint32 are refused before anything is allocated.  The rest of that file needs a device: slabs by the thousand,
cohorts of several GB, torch streams, a second GPU and real allocation failures."""
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))
import test_gpu_king_limits as L
from test_emu_resident import _clone, emu_api  # noqa: F401  (emu_api is a fixture)

test_king_create_refuses_sizes_it_cannot_index_emulated = _clone(L.test_king_create_refuses_sizes_it_cannot_index)
