"""Recorded runs of the tools the host-tool tests compare with, replayed from tests/golden/recorded_runs.json.

The tests were written against the compiled adobe/zdw reference (convertDWfile, unconvertDWfile, test_unconvert_api and
the api_rowloop twin built against its library), which is not part of this repository.  The record in the repository
is a snapshot of this project's own tools, not of the reference: tests/golden/README.md says which commit it was taken
from.  It holds the project to the output it had then; where the reference is built, recording from it turns the
comparison back into one with the reference.

A run is keyed by the tool, its arguments, its stdin and the files in its working directory; the record keeps its exit
code, stdout, stderr and the files under that directory afterwards.  Short stdout / stderr are kept as text; longer
ones and the files as a SHA-256 digest (a `Digest` compares equal to the bytes it was taken from).  A replayed run
leaves nothing in the working directory: its files come back in the result.

ZDW_RECORD_RUNS=DIR starts a new record: the tools in DIR run for real, each in a copy of the working directory, and
what they did replaces the record.  Record with every test of test_host_cli.py and test_gpu_c5.py on a GPU box.
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
RECORD = ROOT / "tests" / "golden" / "recorded_runs.json"
NOCOMP = ROOT / "oracle" / "_ref" / "nocomp"   # gzip / zcat pass-through: the compressor stage is out of scope
TOOL_DIR = b"<tool dir>"                      # stands for the directory of the tool in recorded outputs
INLINE_MAX = 16384


class Digest(str):
    """SHA-256 (hex) of recorded output too long to keep; equal to the bytes it was taken from."""

    def __eq__(self, other):
        if isinstance(other, (bytes, bytearray, memoryview)):
            return hashlib.sha256(other).hexdigest() == str(self)
        return str.__eq__(self, other)

    def __ne__(self, other):
        return not self.__eq__(other)

    __hash__ = str.__hash__

    def _only_equality(self, *a):
        raise AssertionError(f"recorded output over {INLINE_MAX} bytes is kept as its SHA-256 only: compare it with ==")

    __add__ = __radd__ = __contains__ = decode = splitlines = split = _only_equality


def env() -> dict:
    e = dict(os.environ)
    e["PATH"] = f"{NOCOMP}:{e.get('PATH', '')}"
    return e


def files_under(d: Path) -> dict:
    """{path relative to d: bytes} of every file below d."""
    return {p.relative_to(d).as_posix(): p.read_bytes() for p in sorted(d.rglob("*")) if p.is_file()}


def _sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def _key(tool: str, args, cwd: Path, stdin: bytes | None) -> str:
    ins = {k: _sha(v) for k, v in files_under(cwd).items()}
    return _sha(json.dumps([tool, list(args), None if stdin is None else _sha(stdin), ins], sort_keys=True).encode())


def _store(b: bytes, inline_max: int = INLINE_MAX):
    return b.decode("latin1") if len(b) <= inline_max else {"sha256": _sha(b)}


def _load(v):
    return v.encode("latin1") if isinstance(v, str) else Digest(v["sha256"])


_record = None


def _records() -> dict:
    global _record
    if _record is None:
        recording = os.environ.get("ZDW_RECORD_RUNS")
        _record = {} if recording or not RECORD.exists() else json.loads(RECORD.read_text())
    return _record


def run(tool: str, args, cwd: Path, stdin: bytes | None = None, timeout: int = 300):
    """-> (exit code, stdout, stderr, {path under cwd: bytes or Digest}) of the recorded `tool` run in cwd."""
    key = _key(tool, args, cwd, stdin)
    rec = _records()
    tools = os.environ.get("ZDW_RECORD_RUNS")
    if tools:
        tools = Path(tools).resolve()
        with tempfile.TemporaryDirectory(prefix="zdwrec_") as t:
            work = Path(t) / "cwd"
            shutil.copytree(cwd, work)
            p = subprocess.run([str(tools / tool), *args], cwd=work, env=env(), input=stdin, capture_output=True,
                               timeout=timeout)
            norm = lambda b: b.replace(str(tools).encode(), TOOL_DIR)
            rec[key] = {"tool": tool, "args": " ".join(args)[:120], "rc": p.returncode, "stdout": _store(norm(p.stdout)),
                        "stderr": _store(norm(p.stderr)), "files": {k: _store(v, -1) for k, v in files_under(work).items()}}
        RECORD.write_text(json.dumps(rec, indent=0, sort_keys=True) + "\n")
    if key not in rec:
        raise LookupError(f"no recorded run of {tool} {list(args)} on these inputs: record it with "
                          "ZDW_RECORD_RUNS=<directory of the tools> (tests/recorded_runs.py)")
    r = rec[key]
    return r["rc"], _load(r["stdout"]), _load(r["stderr"]), {k: _load(v) for k, v in r["files"].items()}
