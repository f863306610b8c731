"""test_gpu_wide_counts.py under the warp emulator (see test_emu_resident.py): the same checks at a few widths around the
flush points of tier 1, with the product's kernel and C-ABI sources compiled with g++ and "device" buffers in host
memory.  The widths of 100,000 samples and more stay on the GPU."""
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))
import test_gpu_resident as R
import test_gpu_wide_counts as X
from test_emu_resident import emu_api  # noqa: F401  (a fixture)

FLUSH = X.FLUSH


@pytest.fixture
def mem():
    return R.HostMem()


@pytest.mark.parametrize("W", X.WIDTHS)
def test_wide_inputs_are_lossless_at_every_width(oracle, W):
    """The generator's rows at every width of the GPU file, both modes, without a device: each AF row on a rounding edge
    of its mode's formatter, each HWE cohort sensitive to a one-sample move.  (At 98,176 samples int(alt / total * total) in
    float64 is one allele below alt: the edge search starts from the integer count.)"""
    for mode in X.MODES:
        X.self_check(oracle, X.wide_input(oracle, W, mode))


@pytest.mark.parametrize("W", (FLUSH - 1, FLUSH + 32, 2 * FLUSH + 1))
def test_af_hwe_counts_at_width_emulated(emu_api, oracle, mem, W):
    X.check_af_hwe(emu_api, oracle, mem, W)


@pytest.mark.parametrize("W", (2 * FLUSH + 1,))
def test_allele_counter_at_width_emulated(emu_api, oracle, mem, W):
    X.check_allele_counter(emu_api, oracle, mem, W)


@pytest.mark.parametrize("W", (FLUSH + 32,))
def test_dosage_at_width_emulated(emu_api, oracle, mem, W):
    X.check_dosage(emu_api, oracle, mem, W)


@pytest.mark.parametrize("W", (FLUSH + 32,))
def test_inbreeding_at_width_emulated(emu_api, oracle, mem, W):
    X.check_inbreeding(emu_api, oracle, mem, W)


@pytest.mark.parametrize("W", (FLUSH + 1,))
def test_deciding_sample_at_width_emulated(emu_api, oracle, mem, W):
    X.check_deciders(emu_api, oracle, mem, W)
