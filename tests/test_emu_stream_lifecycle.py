"""A stream that fails part-way leaves nothing behind in the context cache (under the warp emulator, see test_emu_parity.py).

The tools keep drained contexts for reuse, keyed by their settings.  A line longer than chunk_bytes is found only when
the chunking reaches it, after the chunks in front of it were submitted.  If the failed stream's context stayed cached
with those chunks in flight, the next call with the same settings would drain them into its own result.  Each case
makes one call fail that way, then makes a call on a good input with the same settings and compares it with the oracle.
"""
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent / "emu"))

CHUNK = 4096


@pytest.fixture(scope="module")
def emu_api():
    import build_emu
    api = build_emu.load_api()
    yield api
    api.close_cached_contexts()


def _inputs():
    from vcfx_b200 import synth
    good = synth.make_vcf(3, 200, 12, seed=29)
    assert len(good) > 4 * CHUNK and max(len(l) for l in good.split(b"\n")) < CHUNK // 4
    cut = good.index(b"\n", 3 * CHUNK) + 1                   # three full chunks come before the long line
    long_line = b"1\t999999\t.\tA\tG\t.\tPASS\t.\tGT" + b"\t0/1" * CHUNK + b"\n"
    return good, good[:cut] + long_line + good[cut:]


TOOLS = {
    "missing_detector": ("missing_detector", "missing"),
    "indexer": ("indexer", "indexer"),
    "nonref_filter": ("nonref_filter", "nonref_filter"),     # goes through the shared helper of the simple tools (control)
}


@pytest.mark.parametrize("mode", [0, 1], ids=["file", "stdin"])
@pytest.mark.parametrize("tool", sorted(TOOLS))
def test_failed_stream_does_not_leak_into_the_next_call(emu_api, oracle, tool, mode):
    fn, ref = (getattr(emu_api, TOOLS[tool][0]), getattr(oracle, TOOLS[tool][1]))
    good, bad = _inputs()
    emu_api.close_cached_contexts()
    with pytest.raises(emu_api.VcfxCudaError, match="longer than chunk_bytes"):
        fn(bad, mode, chunk_bytes=CHUNK)
    assert fn(good, mode, chunk_bytes=CHUNK).out == ref(good, mode).out
