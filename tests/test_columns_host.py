"""Columnar decode, the parts that need no GPU: the file-header reader against the C restatement, the ctypes mirrors of
zdwb_columns_opts / zdwb_columns_out against a C compiler's layout, the library's export and ABI version, and the host
helpers of ColumnBlock / read_columns."""
import bz2
import ctypes as C
import re
import subprocess

import pytest

import corpus
import oracle as O
from test_abi import HEADER


def _images():
    out = [(name, O.golden(name)) for name in ("test.zdw", "analytics-hits.zdw", "movie_tickets.zdw")]
    sch = O.parse_desc(corpus.desc([("a", "varchar(9)"), ("b", "int(11)"), ("c", "char(1)")]))
    tsv = b"x\t1\ty\nzz\t-2\t\\\\\n"
    for md in ({}, {"k": "v"}, {"lineage": "base,2|other,7", "a=": "", "zz": "line\tvalue"}):
        r = O.encode(sch, tsv, metadata=md)
        assert r.rc == 0
        out.append((f"v11_{len(md)}", r.data, md))
    return out


@pytest.mark.parametrize("item", _images(), ids=lambda it: it[0])
def test_read_header_matches_the_c_restatement(item):
    from zdw_b200 import read_header
    image = item[1]
    sch, ver, hl = O.read_header(image)
    h = read_header(image)
    assert (h.version, h.names, h.types, h.charsize, h.length) == (ver, sch.names, sch.types, sch.charsize, hl)
    if ver >= 11:
        assert h.metadata == item[2]
    else:
        assert h.metadata == {}


def test_read_header_rejects_what_is_not_a_header():
    from zdw_b200 import read_header
    with pytest.raises(ValueError):
        read_header(b"\x08\x00a\0\0")  # version 8
    with pytest.raises(ValueError):
        read_header(b"\x0b\x00\xff\x00\x00\x00")  # metadata longer than the file
    with pytest.raises(ValueError):
        read_header(b"\x0a\x00abc")  # names never end


def test_columns_structs_match_the_header_layout(tmp_path):
    from zdw_b200 import capi
    pairs = [("zdwb_columns_opts", capi._ColOpts), ("zdwb_columns_out", capi._ColsOut)]
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    lines = ['#include <stddef.h>', '#include <stdio.h>', f'#include "{HEADER}"', "int main(void) {"]
    fields = {}
    for cname, _ in pairs:
        body = re.search(r"typedef struct\s*\{([^}]*)\}\s*" + cname + r"\s*;", text).group(1)
        names = re.findall(r"([A-Za-z_][A-Za-z0-9_]*)\s*(?:\[[^\]]*\])?\s*;", body)
        fields[cname] = names
        lines.append(f'  printf("{cname} %zu", sizeof({cname}));')
        for f in names:
            lines.append(f'  printf(" %zu", offsetof({cname}, {f}));')
        lines.append('  printf("\\n");')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    for (cname, mirror), line in zip(pairs, out):
        nums = [int(x) for x in line.split()[1:]]
        assert C.sizeof(mirror) == nums[0], cname
        assert [f[0] for f in mirror._fields_] == fields[cname]
        offs = [getattr(mirror, f[0]).offset for f in mirror._fields_]
        assert offs == nums[1:], (cname, fields[cname])


def test_library_exports_decode_columns_at_abi_5():
    from zdw_b200 import capi
    lib = C.CDLL(str(capi.lib_path()))
    assert hasattr(lib, "zdwb_decode_columns")
    assert "zdwb_decode_columns" in capi.EXPORTED_SYMBOLS
    assert capi.load_library().zdwb_abi_version() == 5


def test_column_block_strings_on_the_host():
    import torch
    from zdw_b200 import ColumnBlock
    d = b"\0ab\0b\0zzz\0"
    eo = [1, 4, 6, len(d)]
    vals = torch.tensor([[0, -1, 2, 1], [5, 6, 7, 8]], dtype=torch.int64)
    blk = ColumnBlock(vals, torch.frombuffer(bytearray(d), dtype=torch.uint8), torch.tensor(eo, dtype=torch.int64), [3, 0],
                      4, 0, True, 16384, 2)
    assert blk.strings(0) == [b"ab", None, b"zzz", b"b"]


def test_read_columns_refuses_zstd_and_unknown_names(tmp_path):
    from zdw_b200 import read_columns
    p = tmp_path / "x.zdw.zst"
    p.write_bytes(b"\x28\xb5\x2f\xfd")
    with pytest.raises(ValueError, match="zstd"):
        read_columns(p)
    q = tmp_path / "t.zdw.bz2"
    q.write_bytes(bz2.compress(O.golden("test.zdw")))
    with pytest.raises(KeyError):
        read_columns(q, ["no such column"])
