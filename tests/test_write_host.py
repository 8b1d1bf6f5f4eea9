"""Writing columns back to rows, the parts that need no GPU: the ctypes mirror of zdwb_render_out against a C compiler's
layout, the export and the ABI version, and the pure-Python restatement of the cell texts and the rejection rules
(tests/render_util.py) against the C restatement of the encoder and the decoder (oracle/)."""
import ctypes as C
import random
import re
import subprocess

import oracle as O
import render_util as R
from columns_util import CHAR, INT64_MIN, TEXT_LIKE, UNSIGNED
from columns_util import render as decoder_text
from test_abi import HEADER

ALL_TYPES = sorted(R.KNOWN)


def test_render_out_matches_the_header_layout(tmp_path):
    from zdw_b200 import capi
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    body = re.search(r"typedef struct\s*\{([^}]*)\}\s*zdwb_render_out\s*;", text).group(1)
    names = re.findall(r"([A-Za-z_][A-Za-z0-9_]*)\s*;", body)
    src = tmp_path / "layout.c"
    src.write_text("\n".join(['#include <stddef.h>', '#include <stdio.h>', f'#include "{HEADER}"', "int main(void) {",
                              '  printf("%zu", sizeof(zdwb_render_out));'] +
                             [f'  printf(" %zu", offsetof(zdwb_render_out, {f}));' for f in names] +
                             ['  printf("\\n");', "  return 0;", "}"]))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(src)], check=True)
    nums = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert C.sizeof(capi._RenderOut) == nums[0]
    assert [f[0] for f in capi._RenderOut._fields_] == names
    assert [getattr(capi._RenderOut, f[0]).offset for f in capi._RenderOut._fields_] == nums[1:]


def test_library_exports_render_columns_at_abi_5():
    from zdw_b200 import capi
    lib = C.CDLL(str(capi.lib_path()))
    assert hasattr(lib, "zdwb_render_columns")
    assert "zdwb_render_columns" in capi.EXPORTED_SYMBOLS
    assert capi.load_library().zdwb_abi_version() == 5
    import zdw_b200
    assert "write_table" in zdw_b200.__all__


def _schema(types):
    return O.Schema([f"c{k}" for k in range(len(types))], list(types), [0] * len(types))


def random_string(rng) -> bytes:
    """a string the row reader gives back unchanged: escaped tabs and newlines, backslash pairs, spaces, high bytes"""
    parts = []
    for _ in range(rng.randint(1, 6)):
        parts.append(rng.choice([b"a", b"Zq", b" ", b"  ", b"\\\t", b"\\\n", b"\\\\", b"\xff", b"\x80x", b"0.5", b"-"]))
    s = b"".join(parts)
    return s


def random_cell(rng, t, n_ents):
    if t in TEXT_LIKE:
        return -1 if rng.random() < 0.2 else rng.randrange(n_ents)
    if t == CHAR:
        form = rng.randrange(3)
        if form == 0:
            return 0
        if form == 1:
            return R.sx(rng.choice([b for b in range(1, 256) if b not in (9, 10, 0x5C)]))
        return 0x5C + R.sx(rng.randrange(1, 256)) * 256
    special = [0, 1, -1, INT64_MIN, (1 << 63) - 1, 10, 99, -10]
    if rng.random() < 0.3:
        return rng.choice(special)
    return rng.randrange(-(1 << 63), 1 << 63) >> rng.randrange(64)


def test_rendered_cells_encode_back_to_the_same_cells():
    """The Python-rendered TSV of seeded random cells of every type, encoded and decoded by the C restatement, gives the
    decoder's text of the same cells: the encoder read back every cell."""
    rng = random.Random(11)
    for trial in range(60):
        ncols = rng.choice([1, 2, 5, len(ALL_TYPES)])
        types = ALL_TYPES[:] if ncols == len(ALL_TYPES) else [rng.choice(ALL_TYPES) for _ in range(ncols)]
        ents = sorted({random_string(rng) for _ in range(rng.randint(1, 40))})
        dd = R.make_dict(ents)
        nrows = rng.randint(1, 60)
        cols = [[random_cell(rng, t, len(ents)) for _ in range(nrows)] for t in types]
        dicts = [dd if t in TEXT_LIKE else None for t in types]
        if ncols == 1:  # a one-column row must not render empty
            cols[0] = [v for v in cols[0] if R.cell_text(types[0], v, dd)] or [1 if types[0] not in TEXT_LIKE else 0]
        assert R.check(types, cols, dicts) is None
        tsv = R.render(types, cols, dicts)
        enc = O.encode(_schema(types), tsv)
        assert enc.rc == 0 and enc.total_rows == len(cols[0]), trial
        dec = O.decode(enc.data)
        want = b"".join(b"\t".join(decoder_text(t, v, ents) for t, v in zip(types, row)) + b"\n" for row in zip(*cols))
        assert dec.rc == 0 and dec.tsv == want, trial


def test_writable_holds_exactly_when_the_reader_gives_the_field_back():
    """Over random strings of {a, ' ', \\\\, \\t, \\n, \\xff}: writable(s) iff the C restatement reads s back as the same
    field, as the first, a middle and the last column of a row."""
    rng = random.Random(12)
    alphabet = [b"a", b" ", b"\\", b"\t", b"\n", b"\xff"]
    sch = _schema([0, 1, 0])
    seen = {True: 0, False: 0}
    for _ in range(3000):
        s = b"".join(rng.choice(alphabet) for _ in range(rng.randint(1, 8)))
        tsv = s + b"\tp\tq\n" + b"p\t" + s + b"\tq\n" + b"p\tq\t" + s + b"\n"
        enc = O.encode(sch, tsv)
        back = enc.rc == 0 and enc.total_rows == 3 and O.decode(enc.data).tsv == tsv
        assert R.writable(s) == back, s
        seen[back] += 1
    assert min(seen.values()) > 300


def test_char_forms():
    assert R.char_rule(0) == 0 and R.cell_text(CHAR, 0, None) == b""
    for b in range(1, 256):
        v = R.sx(b)
        assert (R.char_rule(v) == 0) == (b not in (9, 10, 0x5C))
        w = 0x5C + v * 256
        assert R.char_rule(w) == 0 and R.cell_text(CHAR, w, None) == b"\\" + bytes([b])
    for bad in (ord("a") + ord("b") * 256, 0x5C, 9, 10, 128, -129, 0x5C + 128 * 256, 0x5D + 256):
        assert R.char_rule(bad) == R.CHAR_FORM, bad


def test_rejections_name_the_lowest_cell():
    d, eo = R.make_dict([b"ok", b"a\tb", b"x\\", b"y\\\\", b"\\\tz"])
    dd = (d, eo)
    assert R.check([0], [[0, 3, 4, -1]], [dd]) == (0, 3, R.EMPTY_ROW)
    assert R.check([0, 7], [[0, 3, 4, -1], [1, 2, 3, 4]], [dd, None]) is None
    assert R.check([0, 0], [[0, 0, 2], [1, 0, 0]], [dd, dd]) == (0, 2, R.BACKSLASH)
    assert R.check([0, 0], [[0, 0, 0], [0, 1, 0]], [dd, dd]) == (1, 1, R.SEPARATOR)
    assert R.check([0, 6], [[0, 5], [0, 0]], [dd, None]) == (0, 1, R.CODE)
    assert R.check([0, 6], [[0, -2], [0, 0]], [dd, None]) == (0, 1, R.CODE)
    assert R.check([6, 0], [[0, 0x5C], [0, 0]], [None, dd]) == (0, 1, R.CHAR_FORM)
    assert R.check([7, 4], [[1], [1]], [None, None]) == (1, None, None)
    bad = (d[:-1], eo)  # the last entry runs past the dictionary
    assert R.check([0, 7], [[0, 4], [1, 1]], [bad, None]) == (0, 1, R.OFFSETS)
    assert R.check([0, 7], [[0, 0], [1, 1]], [bad, None]) is None  # unreferenced bad entries are fine
    nul = (b"\0a\0b\0c\0", [1, 5, 7])  # entry 0 holds a NUL
    assert R.check([1, 7], [[1, 0], [1, 1]], [nul, None]) == (0, 1, R.ENTRY)
    empty = (b"\0\0x\0", [1, 2, 4])
    assert R.check([1, 7], [[1, 0], [1, 1]], [empty, None]) == (0, 1, R.ENTRY)


def test_signed_and_unsigned_texts():
    assert R.cell_text(15, INT64_MIN, None) == b"-9223372036854775808"
    assert R.cell_text(10, -1, None) == b"18446744073709551615"
    assert R.cell_text(12, 0, None) == b"0" and R.cell_text(7, 0, None) == b"0"
    for t in UNSIGNED | R.SIGNED:
        for v in (0, 1, -1, INT64_MIN, (1 << 63) - 1):
            # strtoull reads the text back to the same 64 bits
            txt = R.cell_text(t, v, None).decode()
            assert (int(txt) & ((1 << 64) - 1)) == (v & ((1 << 64) - 1))
