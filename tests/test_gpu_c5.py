"""Config C5 (BASELINE.json configs[4]): synthetic high-cardinality text, dictionary-bound.  Every text cell is a new
unique 65-byte string, so the block exercises the large-dictionary path (hash set growth, radix sort with tie
refinement, 4-byte offsets) that analytics-shaped data never reaches.  Bit-exact .zdw against the oracle on a prefix,
bit-exact round trip on the whole block, decode through the row-at-a-time C++ API binary."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.gpu
def test_c5_high_cardinality_block():
    p = subprocess.run([sys.executable, str(ROOT / "tests" / "c5_check.py"), "--rows", "400000", "--oracle-rows", "60000"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    assert res["zdw_bit_exact_vs_oracle"] and res["decode_bit_exact_vs_oracle"] and res["roundtrip_bit_exact"]
    assert res["dict_entries"] == 2 * 400000 + 97


@pytest.mark.gpu
def test_c5_decode_through_unconvert_api(tmp_path):
    sys.path.insert(0, str(ROOT / "tests"))
    import c5_check
    import oracle as O
    tsv = c5_check.make_rows(50000)
    z = O.encode(O.parse_desc(c5_check.DESC), tsv, rows_per_block=20000).data  # three blocks
    (tmp_path / "c5.zdw").write_bytes(z)
    import recorded_runs as RR
    p = subprocess.run([str(ROOT / "zdw_b200" / "bin" / "test_unconvert_api"), "c5.zdw"], cwd=tmp_path, capture_output=True,
                       timeout=300)
    assert p.returncode == 0, p.stderr[-500:]
    rc, ref_out, ref_err, _ = RR.run("test_unconvert_api", ["c5.zdw"], tmp_path)
    assert rc == 0, ref_err
    assert p.stdout == ref_out == tsv


@pytest.mark.gpu
@pytest.mark.parametrize("plan", [[(1000, 0), (3000, 0), (9000, 0), (27000, 0)],    # every block longer than the one before: the
                                  [(30000, 0), (6000, 0), (3000, 0), (500, 0)],     # helper's buffer is too short / too long
                                  [(1, 0), (1, 0), (20000, 0), (1, 0)]])
@pytest.mark.parametrize("ahead", [True, False])
def test_unconvert_api_decode_ahead(tmp_path, plan, ahead):
    """getRow over blocks of very different sizes: the block decoded ahead on the helper thread (or, when the helper had
    buffered too little of it, decoded again the ordinary way) gives the rows the one-thread loop gives."""
    import os
    sys.path.insert(0, str(ROOT / "tests"))
    import c5_check
    import oracle as O
    tsv = c5_check.make_rows(50000)
    z = O.encode(O.parse_desc(c5_check.DESC), tsv, plan=plan, rows_per_block=10000)
    assert z.rc == 0 and z.nblocks >= 5
    (tmp_path / "c5.zdw").write_bytes(z.data)
    env = dict(os.environ)
    if not ahead:
        env["ZDW_NO_DECODE_AHEAD"] = "1"
    p = subprocess.run([str(ROOT / "zdw_b200" / "bin" / "test_unconvert_api"), "c5.zdw"], cwd=tmp_path, capture_output=True, timeout=300,
                       env=env)
    assert p.returncode == 0, p.stderr[-500:]
    assert p.stdout == tsv


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["test", "movie_tickets", "analytics-hits"])
def test_api_rowloop_twins_agree_on_goldens(tmp_path, name):
    """The getRow loop (tests/api_rowloop.cpp) built against our host classes and against the unmodified reference
    walks the reference's own golden files to the same rows: same count, same checksum over every field byte."""
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle as O
    (tmp_path / "g.zdw").write_bytes(O.golden(f"{name}.zdw"))
    import recorded_runs as RR
    p = subprocess.run([str(ROOT / "zdw_b200" / "bin" / "api_rowloop"), "--checksum", "g.zdw"], cwd=tmp_path,
                       capture_output=True, timeout=300)
    rc, ref_out, ref_err, _ = RR.run("api_rowloop", ["--checksum", "g.zdw"], tmp_path)
    res = []
    for code, out, err in ((p.returncode, p.stdout, p.stderr), (rc, ref_out, ref_err)):
        assert code == 0, err[-500:]
        res.append(json.loads(out.decode().strip().splitlines()[-1]))
    assert (res[0]["rows"], res[0]["tsv_bytes"], res[0]["fnv1a"]) == (res[1]["rows"], res[1]["tsv_bytes"], res[1]["fnv1a"])
