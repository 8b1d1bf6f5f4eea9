"""Merged dictionaries, the parts that need no GPU: the ctypes mirrors of zdwb_code_part / zdwb_merge_out against a C
compiler's layout, the export and the ABI version, and the host helpers of MergedCodes and ColumnTable."""
import ctypes as C
import re
import subprocess

import pytest

from test_abi import HEADER


def test_merge_structs_match_the_header_layout(tmp_path):
    from zdw_b200 import capi
    pairs = [("zdwb_code_part", capi._CodePart), ("zdwb_merge_out", capi._MergeOut)]
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


def test_library_exports_merge_codes_at_abi_5():
    from zdw_b200 import capi
    lib = C.CDLL(str(capi.lib_path()))
    assert hasattr(lib, "zdwb_merge_codes")
    assert "zdwb_merge_codes" in capi.EXPORTED_SYMBOLS
    assert capi.load_library().zdwb_abi_version() == 5


def _dict(ents):
    import torch
    d = b"\0" + b"".join(e + b"\0" for e in ents)
    eo, at = [], 1
    for e in ents:
        eo.append(at)
        at += len(e) + 1
    eo.append(at)
    return torch.frombuffer(bytearray(d), dtype=torch.uint8), torch.tensor(eo, dtype=torch.int64)


def test_merged_codes_strings_on_the_host():
    import torch
    from zdw_b200 import MergedCodes
    d, eo = _dict([b"", b"ab", b"b\xff"])
    m = MergedCodes(torch.tensor([2, -1, 0, 1, 1], dtype=torch.int64), d, eo)
    assert m.entries == 3
    assert m.strings() == [b"b\xff", None, b"", b"ab", b"ab"]
    empty = MergedCodes(torch.full((3,), -1, dtype=torch.int64), torch.empty(0, dtype=torch.uint8),
                        torch.zeros(1, dtype=torch.int64))
    assert empty.entries == 0 and empty.strings() == [None, None, None]


def test_column_table_strings_on_the_host():
    import torch
    from zdw_b200 import ColumnTable
    d, eo = _dict([b"x", b"yy"])
    vals = torch.tensor([[1, -1, 0], [7, 8, 9]], dtype=torch.int64)
    t = ColumnTable(vals, [(d, eo), None], [4, 0], [2, 1])
    assert t.strings(0) == [b"yy", None, b"x"]
    with pytest.raises(ValueError):
        t.strings(1)


def test_text_like_types_match_the_header():
    """read_table merges exactly the columns that zdwb_decode_columns codes (is_text_like, named in the header)."""
    from zdw_b200 import capi
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    enum = {name: int(v) for name, v in re.findall(r"\bZDWB_([A-Z0-9_]+)\s*=\s*(\d+)", text)}
    names = ["VARCHAR", "TEXT", "DATETIME", "CHAR_2", "DECIMAL", "TINYTEXT", "MEDIUMTEXT", "LONGTEXT"]
    assert capi.TEXT_LIKE_TYPES == {enum[n] for n in names}
