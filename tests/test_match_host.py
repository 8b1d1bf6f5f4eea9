"""Predicates over a dictionary, the parts that need no GPU: the ctypes mirrors of the new structs against a C compiler's
layout, the exports, and the Python restatement of LIKE and lower_bound (tests/match_util.py, the oracle of
tests/test_gpu_match.py) against independent oracles: sqlite's LIKE and bisect over sorted()."""
import bisect
import ctypes as C
import random
import re
import sqlite3
import subprocess

import pytest

import match_util as M
from test_abi import HEADER


def test_match_structs_match_the_header_layout(tmp_path):
    from zdw_b200 import capi
    pairs = [("zdwb_like_opts", capi._LikeOpts), ("zdwb_match_out", capi._MatchOut), ("zdwb_strings", capi._Strings),
             ("zdwb_find_out", capi._FindOut)]
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


def test_library_exports_the_predicates_at_abi_5():
    from zdw_b200 import capi
    lib = C.CDLL(str(capi.lib_path()))
    for name in ("zdwb_match_like", "zdwb_find_strings"):
        assert hasattr(lib, name)
        assert name in capi.EXPORTED_SYMBOLS
    assert capi.load_library().zdwb_abi_version() == 5


def _sqlite_like(db, s: bytes, p: bytes, escape, ignore_case) -> bool:
    db.execute(f"PRAGMA case_sensitive_like={'OFF' if ignore_case else 'ON'}")
    if escape is None:
        return bool(db.execute("SELECT ? LIKE ?", (s.decode(), p.decode())).fetchone()[0])
    return bool(db.execute("SELECT ? LIKE ? ESCAPE ?", (s.decode(), p.decode(), chr(escape))).fetchone()[0])


def _rand_pattern(rng, alphabet, escape):
    lits = bytes(c for c in alphabet if c not in (0x25, 0x5F) and c != escape)
    toks = []
    for _ in range(rng.randint(0, 8)):
        r = rng.random()
        if r < 0.25:
            toks.append(b"%")
        elif r < 0.45:
            toks.append(b"_")
        elif r < 0.6 and escape is not None:
            toks.append(bytes([escape, rng.choice(alphabet + b"%_" + bytes([escape]))]))
        else:
            toks.append(bytes([rng.choice(lits)]))
    return b"".join(toks)


@pytest.mark.parametrize("escape", [0x5C, 0x21, None])
@pytest.mark.parametrize("ignore_case", [False, True])
def test_like_restatement_agrees_with_sqlite(escape, ignore_case):
    """Random ASCII strings and patterns full of '%', '_' and escapes (ASCII only: sqlite's '_' counts UTF-8 characters,
    the restatement's counts bytes)."""
    rng = random.Random(f"{escape}-{ignore_case}")
    db = sqlite3.connect(":memory:")
    alphabet = b"aAbB%_\\!z"
    n_match = 0
    for _ in range(6000):
        s = bytes(rng.choice(alphabet) for _ in range(rng.randint(0, 9)))
        p = _rand_pattern(rng, alphabet, escape)
        if rng.random() < 0.3 and s:  # a pattern cut from the string: more matches
            a = rng.randint(0, len(s))
            p = b"%" + bytes(c for c in s[a:a + 3] if c not in (0x25, 0x5F, 0x5C, 0x21)) + b"%"
        want = _sqlite_like(db, s, p, escape, ignore_case)
        assert M.like(s, p, escape, ignore_case) == want, (s, p, escape, ignore_case)
        n_match += want
    assert n_match > 600


def test_like_restatement_fixed_cases():
    assert M.like(b"", b"") and M.like(b"", b"%") and M.like(b"", b"%%") and not M.like(b"", b"_")
    assert M.like(b"x", b"_") and not M.like(b"xy", b"_") and M.like(b"xy", b"%_")
    assert M.like(b"a%b", b"a\\%b") and not M.like(b"axb", b"a\\%b")
    assert M.like(b"axb", b"a%b", None) and M.like(b"a\\b", b"a\\b", None)
    assert M.like(b"ABC", b"abc", ignore_case=True) and not M.like(b"ABC", b"abc")
    assert M.like(b"\xc4", b"\xc4") and not M.like(b"\xe4", b"\xc4", ignore_case=True)  # only ASCII letters fold
    assert M.like(b"\xc3\xa4", b"__") and not M.like(b"\xc3\xa4", b"_")  # '_' is one byte
    assert M.like(b"abcabd", b"%ab_") and M.like(b"abab", b"ab%ab") and not M.like(b"aba", b"ab%ab")
    with pytest.raises(ValueError):
        M.compile_like(b"ab\\")
    with pytest.raises(ValueError):
        M.compile_like(b"ab!", 0x21)


def test_lower_bound_restatement_agrees_with_bisect():
    rng = random.Random(5)
    for _ in range(300):
        ents = sorted({bytes(rng.choice(b"\x00\x01ab\xff") for _ in range(rng.randint(0, 5))) for _ in range(rng.randint(0, 40))})
        for _ in range(30):
            q = bytes(rng.choice(b"\x00\x01ab\xff") for _ in range(rng.randint(0, 6)))
            assert M.lower_bound(ents, q) == bisect.bisect_left(ents, q)


def test_dict_layout():
    d, eo = M.dict_bytes([b"a", b"", b"bc"])
    assert d == b"\0a\0\0bc\0" and eo == [1, 3, 4, 7]
