"""Host layer (zdw_b200/host): the reference-shaped CLIs and C++ API, differential on the same inputs with the same
flags against recorded runs (recorded_runs.py: written against the compiled reference, replayed from a snapshot of
this project's tools where the reference is not built).  The `gpu` tests exercise the CUDA path end to end through
the binaries; the others cover what needs no device (help text, .desc.sql emission, loud failure without a GPU)."""
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import pytest

import corpus
import oracle as O
import recorded_runs as RR

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "zdw_b200" / "bin"

pytestmark = pytest.mark.skipif(not (BIN / "convertDWfile").exists(), reason="host binaries not built (run __graft_entry__.build())")


def run(tool_dir: Path, tool: str, args, cwd, stdin: bytes | None = None, timeout=300):
    p = subprocess.run([str(tool_dir / tool), *args], cwd=cwd, env=RR.env(), input=stdin, capture_output=True, timeout=timeout)
    return p.returncode, p.stdout, p.stderr


def ours(tool: str, args, cwd, stdin: bytes | None = None, timeout=300):
    """-> (exit code, stdout, stderr, {path under cwd: bytes}) like reference_runs.run"""
    return (*run(BIN, tool, args, cwd, stdin, timeout), RR.files_under(cwd))


class Work:
    def __enter__(self):
        self.d = Path(tempfile.mkdtemp(prefix="zdwhost_"))
        return self.d

    def __exit__(self, *a):
        shutil.rmtree(self.d, ignore_errors=True)


def encode_both(tsv: bytes, desc: bytes, args=(), metadata: bytes | None = None, runners=(ours, RR.run)):
    """-> ((rc, zdw, out, files) ours, (rc, zdw, out, files) recorded)"""
    res = []
    for runner in runners:
        with Work() as d:
            (d / "x.sql").write_bytes(tsv)
            (d / "x.desc.sql").write_bytes(desc)
            if metadata is not None:
                (d / "x.metadata").write_bytes(metadata)
            rc, out, err, files = runner("convertDWfile", [*args, "x.sql"], d)
            res.append((rc, files.get("x.zdw.gz"), (out + err).decode("latin1"), sorted(files)))
    return res


def decode_both(zdw: bytes, args=(), name="x.zdw", runners=(ours, RR.run)):
    res = []
    for runner in runners:
        with Work() as d:
            (d / name).write_bytes(zdw)
            rc, out, err, files = runner("unconvertDWfile", [*args, name], d)
            files.pop(name, None)
            res.append((rc, out, err.decode("latin1"), files))
    return res


def encode_ours(*a, **k):
    """encode_both for our tool alone (flags of this build, which the reference does not know)"""
    return encode_both(*a, runners=(ours,), **k)[0]


def decode_ours(*a, **k):
    return decode_both(*a, runners=(ours,), **k)[0]


def decode_recorded(*a, **k):
    return decode_both(*a, runners=(RR.run,), **k)[0]


# ------------------------------------------------------------------------------------------------ no GPU needed
def test_help_text_matches_reference_except_additions():
    with Work() as d:
        for tool in ("convertDWfile", "unconvertDWfile"):
            mine = run(BIN, tool, ["--help"], d)[1].decode()
            ref = RR.run(tool, ["--help"], d)[1].decode()
            kept = [ln for ln in mine.splitlines() if "(B200 build)" not in ln]
            # the additions are listed in one extra paragraph of the encoder help
            assert [ln for ln in kept if ln.strip()] == [ln for ln in ref.splitlines() if ln.strip() and "(B200 build)" not in ln]
        assert run(BIN, "convertDWfile", ["--version"], d)[1] == RR.run("convertDWfile", ["--version"], d)[1]


def test_cli_argument_errors_match_reference():
    for tool, args in (("convertDWfile", ["--bogus"]), ("convertDWfile", ["-q"]), ("convertDWfile", ["-d"]),
                       ("unconvertDWfile", ["-x", "f"]), ("unconvertDWfile", ["-c"]), ("unconvertDWfile", ["-qq", "f"]),
                       ("unconvertDWfile", ["-c", "a", "-ci", "b", "f"]), ("unconvertDWfile", ["-o", "--metadata", "f"]),
                       ("unconvertDWfile", ["--metadata-values=a,a", "f"]), ("unconvertDWfile", ["nonexistent.zdw"])):
        with Work() as d:  # each run in a directory of its own: nothing left by one run keys or changes the other
            a = run(BIN, tool, args, d)
        with Work() as d:
            b = RR.run(tool, args, d)
        assert a[0] == b[0], (tool, args, a, b)
        assert a[2].replace(str(BIN).encode(), RR.TOOL_DIR) == b[2], (tool, args)


def test_desc_only_needs_no_gpu_and_matches_reference():
    for name in ("test", "analytics-hits"):
        z = O.golden(f"{name}.zdw")
        a, b = decode_both(z, ["-o"])
        assert a[0] == b[0] == 0
        assert a[3]["x.desc.sql"] == b[3]["x.desc.sql"]
        a, b = decode_both(z, ["-q", "-o", "-"])
        assert a[1] == b[1]


def test_missing_files_and_desc_errors_match_reference():
    def both(args, files):
        res = []
        for runner in (ours, RR.run):
            with Work() as d:  # each run in a directory of its own, holding only the inputs
                for name, data in files.items():
                    (d / name).write_bytes(data)
                res.append(runner("convertDWfile", args, d))
        return res
    for args in (["a.sql"], ["a.txt"], ["nofile.sql"]):
        a, b = both(args, {"a.sql": b"1\t2\n"})
        assert a[0] == b[0] == 2
        assert a[2].split(b"\n")[-2] == b[2].split(b"\n")[-2]
    a, b = both(["a.sql"], {"a.sql": b"1\t2\n", "a.desc.sql": b"col_without_type\n"})
    assert a[0] == b[0] == 2 and b"DESC_FILE_MISSING_TYPE_INFO" in a[2]


def _gpu_present():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_gpu_present(), reason="only meaningful on a box without a GPU")
def test_encode_fails_loudly_without_gpu():
    with Work() as d:
        (d / "x.sql").write_bytes(O.golden("test.sql"))
        (d / "x.desc.sql").write_bytes(O.golden("test.desc.sql"))
        rc, out, err = run(BIN, "convertDWfile", ["x.sql"], d)
        assert rc == 2 and b"no CPU path" in err
        assert not (d / "x.zdw.gz").exists()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["test", "analytics-hits", "movie_tickets"])
def test_encode_goldens_bit_exact_and_validated(name):
    tsv, desc = O.golden(f"{name}.sql"), O.golden(f"{name}.desc.sql")
    ours, ref = encode_both(tsv, desc, ["-v"])
    assert ours[0] == 0, ours[2]
    assert ours[1] == ref[1] == O.golden_to_v11(O.golden(f"{name}.zdw"))
    assert "x.zdw.gz GOOD" in ours[2] and f"Rows={tsv.count(10)}" in ours[2]
    assert ours[3] == ref[3]  # same files left behind


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in corpus.cases() if not c[0].startswith("d2_")], ids=lambda c: c[0])
def test_encode_corpus_matches_reference_binary(case):
    name, desc, tsv, opts = case
    args = ["-t"] if opts.get("trim") else []
    ours, ref = encode_both(tsv, desc, args)
    assert ours[0] == ref[0], (name, ours[2], ref[2])
    assert ours[1] == ref[1], name
    if ref[0] != 0:  # error text: "Row N had the problem", internal error code line
        tail = lambda s: [ln for ln in s.splitlines() if "had the problem" in ln or "Internal error" in ln]
        assert tail(ours[2]) == tail(ref[2])
        assert ours[3] == ref[3]  # including the .creating leftover of the wrong-column-count path


@pytest.mark.gpu
def test_metadata_sources_and_precedence():
    tsv, desc = O.golden("test.sql"), O.golden("test.desc.sql")
    for args, mfile in ((["--metadata:b=2", "--metadata:a=1"], None), ([], b"k=v\nlineage=f1,10|f2,20\n"),
                        (["--metadata:cli=wins"], b"file=loses\n")):
        ours, ref = encode_both(tsv, desc, args, mfile)
        assert ours[0] == ref[0] == 0 and ours[1] == ref[1]
    ours, ref = encode_both(tsv, desc, ["--metadata:a=b\nc"])
    assert ours[0] == ref[0] == 2 and ours[1] is None
    ours, ref = encode_both(tsv, desc, [], b"no equals sign\n")
    assert ours[0] == ref[0] == 2
    z = encode_ours(tsv, desc, ["--metadata:b=2", "--metadata:a=1"])[1]
    for args in (["--metadata", "-"], ["--metadata", "--metadata-keys", "-"], ["--metadata", "--metadata-values=a", "-"],
                 ["--metadata", "--metadata-values=zz", "-"], ["--metadata", "--metadata-values-allow-missing=zz,a", "-"], []):
        a, b = decode_both(z, ["-q", *args])
        assert a[0] == b[0] and a[1] == b[1] and a[3] == b[3], args


@pytest.mark.gpu
def test_streaming_stdin_encode_matches_file_mode():
    tsv, desc = O.golden("test.sql") * 50, O.golden("test.desc.sql")
    want = encode_ours(tsv, desc)[1]
    with Work() as d:
        (d / "x.desc.sql").write_bytes(desc)
        rc, out, err = run(BIN, "convertDWfile", ["-i", "-v", "x.sql"], d, stdin=tsv)
        assert rc == 0, err
        assert (d / "x.zdw.gz").read_bytes() == want
        assert b"GOOD" in out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["test", "analytics-hits", "movie_tickets"])
def test_decode_goldens_all_versions(name):
    z = O.golden(f"{name}.zdw")  # v9 / v10 as shipped by the reference
    for image in (z, O.golden_to_v11(z)):
        a, b = decode_both(image, ["-q"])
        assert a[0] == b[0] == 0, a[2]
        assert a[3]["x.sql"] == O.golden(f"{name}.sql")
        assert a[3] == b[3]  # x.sql and x.desc.sql (and no .metadata)
    a, b = decode_both(z, ["-q", "-"])
    assert a[1] == b[1] == O.golden(f"{name}.sql")
    a, b = decode_both(z, ["-t"])
    assert a[0] == b[0] == 0 and a[1] == b[1] and b"tested good" in a[1]


@pytest.mark.gpu
def test_decode_column_selection_and_virtual_columns():
    z = O.golden("analytics-hits.zdw")
    names = [ln.split(b"\t")[0].decode() for ln in O.golden("analytics-hits.desc.sql").splitlines()]
    some = ",".join([names[700], names[3], names[1500], names[0]])
    for args in (["-c", some], ["-ci", some + ",nope," + names[3].upper()], ["-ce", "nope," + some + ",nada"],
                 ["-cx", ",".join(names[5:2000])], ["-c", "virtual_export_row," + names[0] + ",virtual_export_basename"],
                 ["-ci", "VIRTUAL_EXPORT_ROW,nope"], ["-c", "nope"], ["-ci", "nope,nada"], ["-c", names[0] + "," + names[0]]):
        a, b = decode_both(z, ["-q", *args, "-"])
        assert a[0] == b[0], (args, a[2], b[2])
        assert a[1] == b[1], args
        a, b = decode_both(z, ["-q", *args])
        assert a[0] == b[0] and a[3] == b[3], args
    t = O.golden_to_v11(O.golden("test.zdw"))
    for args in (["--non-empty-column-header"], ["--non-empty-column-header", "-cx", "age"], ["-a", ".bak"], ["-w"], ["-a", ".x", "-w"]):
        a, b = decode_both(t, ["-q", *args])
        assert a[0] == b[0] == 0 and a[3] == b[3], args


@pytest.mark.gpu
def test_decode_stdin_and_output_dir():
    z = O.golden_to_v11(O.golden("test.zdw"))
    for runner in (ours, RR.run):
        with Work() as d:
            (d / "o").mkdir()
            rc, out, err, files = runner("unconvertDWfile", ["-q", "-i"], d, stdin=z)
            assert rc == 0 and out == O.golden("test.sql")
            rc, out, err, files = runner("unconvertDWfile", ["-q", "-i", "-d", "o/", "named"], d, stdin=z)
            assert rc == 0 and files["o/named.sql"] == O.golden("test.sql")
            assert "o/named.desc.sql" in files


@pytest.mark.gpu
def test_multi_block_files_and_statistics():
    tsv, desc = O.golden("movie_tickets.sql"), O.golden("movie_tickets.desc.sql")
    ours = encode_ours(tsv, desc, ["--rows-per-block=100000"])
    assert ours[0] == 0 and "block 6 of" in ours[2]
    z = ours[1]
    want = O.encode(O.parse_desc(desc), tsv, rows_per_block=100000)
    assert z == want.data and want.nblocks == 6
    a, b = decode_both(z, ["-q", "-"])           # the reference decodes our multi-block file
    assert a[0] == b[0] == 0 and a[1] == b[1] == tsv
    a, b = decode_both(z, ["-s"])
    assert a[0] == b[0] == 0 and a[1] == b[1]      # version, line length, dictionary sizes, equality-bit statistics
    a, b = decode_both(z, ["-t", "-v"])
    assert a[0] == b[0] == 0
    a, b = decode_both(z, ["-q", "-c", "virtual_export_row", "-"])
    assert a[1] == b[1]                            # row numbers run on across blocks
    small = encode_ours(tsv[: 1 << 20].rsplit(b"\n", 1)[0] + b"\n", desc, ["--block-bytes=70000"])
    assert small[0] == 0
    back = decode_both(small[1], ["-q", "-"])
    assert back[0][1] == back[1][1] == tsv[: 1 << 20].rsplit(b"\n", 1)[0] + b"\n"


def _window_plan(tsv: bytes, window: int):
    """[(rows, 0)] for every block but the last when blocks are cut by an input window of `window` bytes: a block
    holds the complete rows of its window, the next window starts behind them (data without escapes)."""
    plan, pos = [], 0
    while pos + window <= len(tsv):
        cut = tsv[pos:pos + window].rfind(b"\n") + 1
        assert cut > 0
        if pos + cut == len(tsv):
            break  # the rows end with this window: it is the last block
        plan.append((tsv[pos:pos + cut].count(b"\n"), 0))
        pos += cut
    return plan


@pytest.mark.gpu
@pytest.mark.parametrize("window", [70000, 131072])
def test_block_bytes_windows_cut_like_the_sequential_loop(window):
    """--block-bytes on a file of many windows: the read-ahead thread, the pinned double buffer and the writer thread
    of convertDWfile must leave the cuts where a plain fill-encode-consume loop puts them; the file must be the one
    the restatement writes for those cuts."""
    tsv = O.golden("movie_tickets.sql")[: 1 << 20].rsplit(b"\n", 1)[0] + b"\n"
    desc = O.golden("movie_tickets.desc.sql")
    ours = encode_ours(tsv, desc, [f"--block-bytes={window}"])
    assert ours[0] == 0, ours[2]
    plan = _window_plan(tsv, window)
    want = O.encode(O.parse_desc(desc), tsv, plan=plan)
    assert want.nblocks == len(plan) + 1 >= 8
    assert ours[1] == want.data


@pytest.mark.gpu
def test_truncated_and_trailing_garbage():
    z = O.golden_to_v11(O.golden("movie_tickets.zdw"))
    a, b = decode_both(z + b"x", ["-q"])   # the final one-byte dummy read swallows a single stray byte
    assert a[0] == b[0] == 0
    a, b = decode_both(z + b"xy", ["-q"])
    assert a[0] == b[0] == 6 and b"Did not reach EOF" in a[1]
    a, b = decode_both(z[: len(z) // 2], ["-q"])   # cut inside the dictionary: the short read throws GZREAD_FAILED,
    assert a[0] == b[0] == -6                       # which neither CLI catches (reference UnconvertFromZDW.cpp:294-300)
    assert "failed" in a[2] and "failed" in b[2]
    a = decode_ours(z[: len(z) - 1000], ["-q"])  # cut inside the rows
    assert a[0] == 8  # ROW_COUNT_ERR (the reference dies on the short read here as well)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["test", "analytics-hits", "movie_tickets"])
def test_unconvert_api_matches_reference(name):
    z = O.golden(f"{name}.zdw")
    for runner in (ours, RR.run):
        with Work() as d:
            (d / "x.zdw").write_bytes(z)
            rc, out, err, _ = runner("test_unconvert_api", ["x.zdw"], d)
            assert rc == 0, err
            assert out == O.golden(f"{name}.sql")
    names = [ln.split(b"\t")[0].decode() for ln in O.golden(f"{name}.desc.sql").splitlines()]
    sel = ",".join([names[-1], "nope", names[0]])
    outs = []
    for runner in (ours, RR.run):
        with Work() as d:
            (d / "x.zdw").write_bytes(z)
            outs.append(runner("test_unconvert_api", ["-ci", sel, "x.zdw"], d)[:2])
    assert outs[0] == outs[1]


@pytest.mark.gpu
def test_block_plan_flag_reproduces_the_references_memory_cut():
    """convertDWfile --block-plan=rows:spill with the plan recovered from the memory-cut file (test_block_plan.memory_cut_file:
    the restatement's file for the cut the reference makes under --mem-limit=140)."""
    import c5_check
    import test_block_plan as BP
    sch = O.parse_desc(c5_check.DESC)
    tsv, image = BP.memory_cut_file()
    plan = BP.recover_plan(sch, tsv, image)
    with Work() as d:
        (d / "x.sql").write_bytes(tsv)
        (d / "x.desc.sql").write_bytes(c5_check.DESC)
        flag = "--block-plan=" + ",".join(f"{r}:{s}" for r, s in plan)
        rc, out, err = run(BIN, "convertDWfile", ["-q", flag, "--block-bytes=16777216", "x.sql"], d, timeout=600)
        assert rc == 0, (out + err)[-500:]
        assert (d / "x.zdw.gz").read_bytes() == image


# ------------------------------------------------------------------------------------------------ block fan-out (SURVEY 8(e))
def _gpu_count():
    try:
        from zdw_b200.capi import load_library
        return load_library().zdwb_device_count()
    except Exception:  # noqa: BLE001
        return 0


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [["--lanes-per-gpu=1"], ["--gpus=0,0", "--lanes-per-gpu=3"], ["--gpus=0,0,0"]])
def test_encode_workers_write_the_sequential_file(flags):
    """Whole blocks dealt out to several encode workers (here: several contexts on device 0): the windows are cut on the
    host before any block is encoded, the blocks leave in file order - same bytes as the one-context loop
    (--lanes-per-gpu=1) and as the restatement for those cuts."""
    tsv = O.golden("movie_tickets.sql")[: 3 << 20].rsplit(b"\n", 1)[0] + b"\n"
    desc = O.golden("movie_tickets.desc.sql")
    ours = encode_ours(tsv, desc, ["--block-bytes=131072", *flags])
    assert ours[0] == 0, ours[2]
    plan = _window_plan(tsv, 131072)
    want = O.encode(O.parse_desc(desc), tsv, plan=plan)
    assert want.nblocks == len(plan) + 1 >= 20
    assert ours[1] == want.data
    assert "Rows=%d" % want.total_rows in ours[2]


@pytest.mark.gpu
def test_encode_workers_report_the_first_bad_row():
    """A malformed row in a later window: exit code 2, the reference's message, the .creating file stays (App. B-19)."""
    rows = [b"%d\tabc\t%d" % (i, i * 3) for i in range(40000)]
    rows[31000] = b"1\t2"
    tsv = b"\n".join(rows) + b"\n"
    desc = corpus.desc([("a", "int(11)"), ("b", "varchar(8)"), ("c", "int(11)")])
    for flags in (["--lanes-per-gpu=1"], ["--gpus=0,0"]):
        ours = encode_ours(tsv, desc, ["--block-bytes=65536", *flags])
        assert ours[0] == 2, ours[2]
        assert "had the problem" in ours[2] and "WRONG_NUM_OF_COLUMNS_ON_A_ROW" in ours[2]
        assert "x.creating.zdw.gz" in ours[3] and "x.zdw.gz" not in ours[3]


@pytest.mark.gpu
def test_c4_file_on_two_gpus_equals_one_gpu_and_the_oracle():
    """>= 16 blocks of C4-shaped rows: --gpus=2 (two real devices; below two GPUs the second worker group shares device
    0) writes the bytes of --gpus=1 and of the restatement, and the reference decodes them to the source rows."""
    import ctypes as C

    import bench
    synth = bench.Synth()
    rows = 1024
    cap = synth.cap_for(rows)
    buf = (C.c_uint8 * cap)()
    parts = []
    for b in range(18):
        n = synth.block_into(40 + b, rows, C.addressof(buf), cap)
        parts.append(bytes(memoryview(buf)[:n]))
    tsv = b"".join(parts)
    window = len(tsv) // 17
    two = "--gpus=2" if _gpu_count() >= 2 else "--gpus=0,0"
    one = encode_ours(tsv, synth.desc, [f"--block-bytes={window}", "--gpus=1", "--lanes-per-gpu=1"])
    par = encode_ours(tsv, synth.desc, [f"--block-bytes={window}", two])
    assert one[0] == 0 and par[0] == 0, one[2] + par[2]
    assert one[1] == par[1]
    plan = _window_plan(tsv, window)
    want = O.encode(O.parse_desc(synth.desc), tsv, plan=plan)
    assert want.nblocks >= 16 and par[1] == want.data
    with Work() as d:
        (d / "x.zdw").write_bytes(par[1])
        rc, ref_tsv, err, _ = RR.run("unconvertDWfile", ["-q", "-", "x.zdw"], d, timeout=600)
    assert rc == 0 and ref_tsv == tsv, err


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [["--lanes-per-gpu=1"], ["--gpus=0,0", "--lanes-per-gpu=2"], ["--lanes-per-gpu=3"]])
def test_decode_workers_write_the_sequential_rows(flags):
    """Blocks skimmed for their length by the calling thread and decoded by several workers: to a regular file (blocks
    written side by side at their offsets) and to stdout (in order through the pipe) - the rows of the one-context
    loop, the reference's rows, column selection and the block header lines included."""
    tsv = O.golden("movie_tickets.sql")[: 3 << 20].rsplit(b"\n", 1)[0] + b"\n"
    desc = O.golden("movie_tickets.desc.sql")
    img = O.encode(O.parse_desc(desc), tsv, rows_per_block=2500)
    assert img.nblocks >= 15
    a = decode_ours(img.data, ["-q", *flags])
    b = decode_recorded(img.data, ["-q"])
    assert a[0] == b[0] == 0, a[2]
    assert a[3]["x.sql"] == b[3]["x.sql"] == tsv
    with Work() as d:
        (d / "x.zdw").write_bytes(img.data)
        rc, out, err = run(BIN, "unconvertDWfile", ["-q", *flags, "-", "x.zdw"], d)
        assert rc == 0 and out == tsv, err
        rc, out, err = run(BIN, "unconvertDWfile", ["-q", *flags, "-c", "revenue,virtual_export_row,movie", "--non-empty-column-header", "-", "x.zdw"], d)
        rc2, out2, err2, _ = RR.run("unconvertDWfile", ["-q", "-c", "revenue,virtual_export_row,movie", "--non-empty-column-header", "-", "x.zdw"], d)
        assert rc == rc2 == 0 and out == out2, err


@pytest.mark.gpu
def test_decode_workers_stop_at_a_corrupt_block():
    """A block cut short in the middle of a multi-block file: same exit code and message as the one-context loop; the
    rows in front of the bad block are written, nothing behind it."""
    tsv = O.golden("movie_tickets.sql")[: 1 << 20].rsplit(b"\n", 1)[0] + b"\n"
    desc = O.golden("movie_tickets.desc.sql")
    img = O.encode(O.parse_desc(desc), tsv, rows_per_block=2500).data
    offs = O.decode(img).block_offset
    cut = img[: offs[4] + (offs[5] - offs[4]) * 7 // 8]  # inside the rows of block 4 (a cut inside a header ends in the
    res = []                                             # reference's uncaught ZDWException instead, SURVEY 8(b))
    for flags in (["--lanes-per-gpu=1"], ["--gpus=0,0"]):
        with Work() as d:
            (d / "x.zdw").write_bytes(cut)
            rc, out, err = run(BIN, "unconvertDWfile", ["-q", *flags, "x.zdw"], d)
            res.append((rc, (d / "x.sql").read_bytes() if (d / "x.sql").exists() else None))
    assert res[0][0] == res[1][0] == 8  # ROW_COUNT_ERR
    assert res[0][1] == res[1][1] == b"".join(tsv.split(b"\n")[k] + b"\n" for k in range(4 * 2500))


@pytest.mark.gpu
def test_c4_file_decodes_on_two_gpus():
    import ctypes as C

    import bench
    synth = bench.Synth()
    rows = 1024
    cap = synth.cap_for(rows)
    buf = (C.c_uint8 * cap)()
    parts = []
    for b in range(17):
        n = synth.block_into(70 + b, rows, C.addressof(buf), cap)
        parts.append(bytes(memoryview(buf)[:n]))
    tsv = b"".join(parts)
    img = O.encode(O.parse_desc(synth.desc), tsv, rows_per_block=rows)
    assert img.nblocks == 17
    two = "--gpus=2" if _gpu_count() >= 2 else "--gpus=0,0"
    a = decode_ours(img.data, ["-q", two])
    b = decode_recorded(img.data, ["-q"])
    assert a[0] == 0, a[2]
    assert a[3]["x.sql"] == tsv == b[3]["x.sql"]


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [["-i", "-v"], ["-i", "-t", "-v"]])
def test_streaming_validation_compares_normalised_rows(flags):
    """-i -v keeps the streamed rows for the round-trip check the way the reference does (GetDataRow,
    ConvertToZDW.cpp:274-283,316-319): blank lines skipped, an unterminated last line dropped, and with -t the fields
    without their trailing spaces - so a good file is reported GOOD, as by the reference (several windows here)."""
    desc = corpus.desc([("a", "varchar(16)"), ("b", "int(11)"), ("c", "varchar(16)")])
    rows = []
    for i in range(5000):
        rows.append(b"name%d   \t%d\tx y \n" % (i % 37, i + 1) if "-t" in flags else b"name%d\t%d\tx y\n" % (i % 37, i + 1))
        if i % 500 == 0:
            rows.append(b"\n\n")
    tsv = b"".join(rows) + b"tail\t1"
    outs = []
    for runner in (ours, RR.run):
        with Work() as d:
            (d / "x.desc.sql").write_bytes(desc)
            extra = ["--block-bytes=20000"] if runner is ours else []
            rc, out, err, files = runner("convertDWfile", [*flags, *extra, "x.sql"], d, stdin=tsv)
            outs.append((rc, b"GOOD" in out, sorted(files), (out + err).decode("latin1")))
    assert outs[0][:3] == outs[1][:3], outs
    assert outs[0][0] == 0 and outs[0][1], outs[0][3]


@pytest.mark.gpu
def test_heap_blocks_flag_reproduces_the_references_memory_cut_without_a_plan():
    """convertDWfile --heap-blocks=2 writes the memory-cut file (the restatement's file for the cut the compiled reference
    makes on its own under --mem-limit=140, test_block_plan.memory_cut_file; K = 2 is
    the allocation at which that process was over its limit, tests/test_block_plan.py) - no explicit plan given.
    --mem-limit itself is accepted and changes nothing."""
    import c5_check
    import test_block_plan as BP
    tsv, image = BP.memory_cut_file()
    with Work() as d:
        (d / "x.sql").write_bytes(tsv)
        (d / "x.desc.sql").write_bytes(c5_check.DESC)
        rc, out, err = run(BIN, "convertDWfile", ["-q", "--heap-blocks=2", "--mem-limit=140", "x.sql"], d, timeout=600)
        assert rc == 0, (out + err)[-500:]
        assert (d / "x.zdw.gz").read_bytes() == image
        # a window smaller than the block: it is widened until heap block 2 opens inside it
        os.unlink(d / "x.zdw.gz")
        rc, out, err = run(BIN, "convertDWfile", ["-q", "--heap-blocks=2", "--block-bytes=8388608", "x.sql"], d, timeout=600)
        assert rc == 0, (out + err)[-500:]
        assert (d / "x.zdw.gz").read_bytes() == image
