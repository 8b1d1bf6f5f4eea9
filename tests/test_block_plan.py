"""Explicit block plan with the reference's interrupted-row spill (SURVEY App. B-14, hard part #3).

The reference closes a block when its process runs low on memory; the row being parsed at that moment is not counted,
but the columns already parsed have fed the dictionary and the column ranges.  (rows, spilled columns) per block is
all it takes to reproduce such a file: the oracle restatement takes them as an explicit plan, and this test recovers
the plan from a file the compiled reference cut on its own (--mem-limit) and checks that the restatement then writes
the same bytes.  The GPU twin of this test (test_gpu_encode.py) holds the CUDA encoder to the same files."""
import functools
import hashlib
import json
import os
import subprocess
import tempfile

import pytest

import c5_check
import corpus
import oracle as O

needs_ref = pytest.mark.skipif(not O.have_ref(), reason="compiled reference (oracle/_ref) not available")


@functools.lru_cache(maxsize=2)
def reference_mem_limit_file(rows: int, mem_limit_mb: int):
    """C5-shaped rows (every text cell a new 65-byte string) through the reference with --mem-limit: (tsv, image)."""
    tsv = c5_check.make_rows(rows)
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
        open(os.path.join(d, "x.sql"), "wb").write(tsv)
        open(os.path.join(d, "x.desc.sql"), "wb").write(c5_check.DESC)
        env = dict(os.environ, PATH=str(O.REF_DIR / "nocomp") + os.pathsep + os.environ["PATH"])
        p = subprocess.run([str(O.REF_DIR / "convertDWfile"), "-q", f"--mem-limit={mem_limit_mb}", "x.sql"], cwd=d, env=env,
                           capture_output=True, timeout=600)
        assert p.returncode == 0, p.stderr[-500:]
        return tsv, open(os.path.join(d, "x.zdw.gz"), "rb").read()


@functools.lru_cache(maxsize=1)
def memory_cut_file():
    """(tsv, image): the rows of tests/golden/memory_cut.json and the file the restatement writes for them with the cut
    kept there (its heap-block model at K = 2, the reference's cut under --mem-limit=140: test_stored_cut_is_the_references),
    checked against the stored SHA-256."""
    cut = json.loads((O.GOLDEN / "memory_cut.json").read_text())
    tsv = c5_check.make_rows(cut["rows"])
    image = O.encode(O.parse_desc(c5_check.DESC), tsv, plan=[tuple(b) for b in cut["plan"]]).data
    assert hashlib.sha256(image).hexdigest() == cut["sha256"]
    return tsv, image


def recover_plan(sch, tsv: bytes, image: bytes):
    """[(rows, spill)] for every block but the last, found block by block: the spill count is the one that makes the
    restatement reproduce the reference's block."""
    ref = O.decode(image)
    assert ref.rc == 0 and ref.nblocks <= 16
    plan = []
    for k in range(ref.nblocks - 1):
        end = ref.block_offset[k + 1]
        for spill in range(sch.ncols + 1):
            got = O.encode(sch, tsv, plan=plan + [(ref.block_rows[k], spill)]).data
            if got[:end] == image[:end]:
                plan.append((ref.block_rows[k], spill))
                break
        else:
            raise AssertionError(f"no spill count reproduces block {k}")
    return plan


@needs_ref
def test_stored_cut_is_the_references():
    assert memory_cut_file() == reference_mem_limit_file(600_000, 140)


@needs_ref
def test_restatement_reproduces_a_memory_cut_file():
    sch = O.parse_desc(c5_check.DESC)
    tsv, image = reference_mem_limit_file(600_000, 140)
    ref = O.decode(image)
    assert ref.nblocks >= 2, "the reference did not cut the file: raise the row count or lower --mem-limit"
    plan = recover_plan(sch, tsv, image)
    assert any(spill for _, spill in plan), plan  # the cut falls inside a row: some columns have been parsed already
    assert O.encode(sch, tsv, plan=plan).data == image
    assert ref.tsv == tsv


@needs_ref
def test_heap_block_model_places_the_references_cut():
    """SURVEY 8f-1 / App. B-14: where the reference cuts a file is a function of the input and ONE number - the
    string-heap allocation at which its process is found over --mem-limit.  The restatement packs new strings into
    64 MiB heap blocks like StringHeap does and ends the ZDW block on the K-th allocation; some small K must reproduce
    the file the reference cut on its own, rows, spilled columns and all."""
    sch = O.parse_desc(c5_check.DESC)
    tsv, image = reference_mem_limit_file(600_000, 140)
    assert O.decode(image).nblocks >= 2
    hits = [k for k in range(1, 7) if O.encode(sch, tsv, heap_blocks=k).data == image]
    assert len(hits) == 1, hits
    # the same cut expressed as an explicit plan
    plan = recover_plan(sch, tsv, image)
    assert O.encode(sch, tsv, plan=plan).data == O.encode(sch, tsv, heap_blocks=hits[0]).data
    # K = 1: the very first string already finds the process over its limit (ConvertToZDW.cpp:824-834)
    assert O.encode(sch, tsv[:100_000].rsplit(b"\n", 1)[0] + b"\n", heap_blocks=1).rc == 7  # OUT_OF_MEMORY


def test_heap_block_model_many_blocks_round_trip():
    sch = O.parse_desc(c5_check.DESC)
    tsv = c5_check.make_rows(1_300_000)   # ~170 MB of new strings: K = 2 closes a block at every 64 MiB of them
    z = O.encode(sch, tsv, heap_blocks=2)
    dec = O.decode(z.data)
    assert z.rc == 0 and dec.rc == 0 and dec.nblocks == z.nblocks >= 3
    assert dec.tsv == tsv


@pytest.mark.parametrize("plan", [[(1000, 0)], [(1000, 3), (500, 1)], [(7, 8)], [(2999, 2)]])
def test_plan_round_trips_on_the_mixed_corpus(plan):
    case = next(c for c in corpus.cases() if c[0] == "mixed_3000")
    sch = O.parse_desc(case[1])
    z = O.encode(sch, case[2], plan=plan)
    dec = O.decode(z.data)
    assert dec.rc == 0 and dec.nblocks == len(plan) + 1
    assert dec.block_rows[:len(plan)] == [r for r, _ in plan]
    assert dec.tsv == O.decode(O.encode(sch, case[2]).data).tsv
