"""The reference tools' side of the CLI comparisons: `run(tool, args, stdin)` gives what `VCFX_<tool> args` prints.

Where the unmodified reference tools are built (oracle/_ref/VCFX_*, `make -C oracle ref REFERENCE=<VCFX source tree>`)
they are run.  Elsewhere the answer comes from tests/golden/recorded_runs.json.gz, which is NOT the reference's own
output: it was recorded from this project's drop-in tools (the emulator build, tests/emu/), at a state of the tools
that matched the reference tools byte for byte on these invocations (the GPU suite of that state ran against
oracle/_ref).  Without a reference build the comparisons therefore pin the drop-in tools, and through
test_oracle_golden the oracle, to that recorded state; the independent pin of the oracle to the reference stays
tests/golden/reference_outputs.json, made from the reference tools themselves.

The table maps one invocation — the tool, its arguments, the bytes on stdin (for a gzip stream: a marker and the
payload) and the bytes of every file named on the command line — to the exit code, the SHA-256 of stdout and the stderr
text.  A file's path is stored as a placeholder wherever it appears in the output, and so is the recording
executable's own path (getopt prints argv[0]).  For allele_counter -z / --gzip the stdout given back, live or recorded,
is the payload of the gzip stream: the container may differ between zlib builds.

To record: run the tests that call `run` with VCFX_RECORD_REFERENCE set to a directory of VCFX_* executables (the
reference build, where there is one), in one process (no -n), on a machine with at least two GPUs so that
test_gpu_cli.py::test_multi_gpu_same_bytes runs too; what each invocation printed is added to the table at exit."""
from __future__ import annotations

import atexit
import gzip
import hashlib
import json
import os
import subprocess
from pathlib import Path

import pytest

PATH = Path(__file__).resolve().parent / "golden" / "recorded_runs.json.gz"
REF_DIR = Path(__file__).resolve().parent.parent / "oracle" / "_ref"
RECORD = os.environ.get("VCFX_RECORD_REFERENCE")
_table: dict | None = None
_recorded: list[str] = []


def _sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def _load() -> dict:
    global _table
    if _table is None:
        _table = json.loads(gzip.decompress(PATH.read_bytes())) if PATH.exists() else {}
    return _table


def _files(args) -> dict[int, str]:
    return {i: a for i, a in enumerate(args) if os.path.isabs(a) and os.path.isfile(a)}


def _key(tool: str, args, stdin: bytes) -> str:
    files = _files(args)
    parts = [tool] + [("file:" + _sha(Path(a).read_bytes())) if i in files else ("arg:" + a) for i, a in enumerate(args)]
    # a gzip stream on stdin is known by its payload: its deflate bytes depend on the zlib build that made it
    parts.append(("stdin-gzip:" + _sha(gzip.decompress(stdin))) if stdin[:2] == b"\x1f\x8b" else ("stdin:" + _sha(stdin)))
    return _sha("\0".join(parts).encode())[:32]


def _gzip_out(tool: str, args) -> bool:
    return tool == "allele_counter" and ("-z" in args or "--gzip" in args)


def _exec(exe: Path, tool: str, args, stdin: bytes):
    """Runs exe; stdout and stderr with exe's path and every file argument's path replaced by placeholders."""
    r = subprocess.run([str(exe), *args], input=stdin, capture_output=True, timeout=600)
    subs = [(str(exe).encode(), exe.name.encode())] + [(a.encode(), b"\0FILE%d\0" % i) for i, a in _files(args).items()]
    out, err = r.stdout, r.stderr
    for real, ph in subs:
        out, err = out.replace(real, ph), err.replace(real, ph)
    return r.returncode, (gzip.decompress(out) if _gzip_out(tool, args) else out), err


def _restore(b: bytes, args) -> bytes:
    for i, a in _files(args).items():
        b = b.replace(b"\0FILE%d\0" % i, a.encode())
    return b


class Stdout:
    """A recorded stdout, known by its digest: equal to the bytes that have the same digest (file paths as placeholders)."""

    def __init__(self, digest: str, args):
        self.digest, self._args = digest, args

    def __eq__(self, other):
        if not isinstance(other, (bytes, bytearray)):
            return NotImplemented
        b = bytes(other)
        for i, a in _files(self._args).items():
            b = b.replace(a.encode(), b"\0FILE%d\0" % i)
        return _sha(b) == self.digest

    def __ne__(self, other):
        r = self.__eq__(other)
        return r if r is NotImplemented else not r

    __hash__ = None

    def __repr__(self):
        return f"<recorded stdout sha256 {self.digest[:16]}>"


def _save():
    PATH.write_bytes(gzip.compress(json.dumps(_table, sort_keys=True, separators=(",", ":")).encode(), 9, mtime=0))


def run(tool: str, args, stdin: bytes | None = None):
    """(exit code, stdout, stderr bytes) of `VCFX_<tool> args` with `stdin` on the reference side: stdout is bytes when
    a reference build ran, a Stdout (compares equal to the same bytes) when it comes from the recorded table."""
    args = [str(a) for a in args]
    stdin = stdin if stdin is not None else b""
    if RECORD:
        rc, out, err = _exec(Path(RECORD).resolve() / f"VCFX_{tool}", tool, args, stdin)
        if not _recorded:
            atexit.register(_save)
        key = _key(tool, args, stdin)
        _recorded.append(key)
        _load()[key] = [rc, _sha(out), err.decode("latin-1")]
        return rc, _restore(out, args), _restore(err, args)
    if (REF_DIR / f"VCFX_{tool}").exists():
        rc, out, err = _exec(REF_DIR / f"VCFX_{tool}", tool, args, stdin)
        return rc, _restore(out, args), _restore(err, args)
    table, key = _load(), _key(tool, args, stdin)
    if key not in table:
        pytest.fail(f"no recorded output for VCFX_{tool} {' '.join(args)} (stdin: {len(stdin)} bytes) and no reference "
                    f"build in oracle/_ref; record it with VCFX_RECORD_REFERENCE=<directory of VCFX_* tools>")
    rc, digest, err = table[key]
    return rc, Stdout(digest, args), _restore(err.encode("latin-1"), args)
