"""A pure-Python restatement of zdwb_render_columns (include/zdw_b200.h): the text of every cell, and the rules by which a
table is refused, for tests/test_write_host.py and tests/test_gpu_write.py."""
from __future__ import annotations

from columns_util import CHAR, TEXT_LIKE, UNSIGNED

SIGNED = {12, 13, 14, 15}
KNOWN = TEXT_LIKE | UNSIGNED | SIGNED | {CHAR}
INT64_MIN = -(1 << 63)

# the rules, numbered as render.cu numbers them
OFFSETS, ENTRY, SEPARATOR, BACKSLASH, CODE, CHAR_FORM, EMPTY_ROW = 1, 2, 3, 4, 5, 6, 7
# words of each rule in zdwb_last_error
RULE_WORDS = {OFFSETS: "offsets", ENTRY: "empty, holds a NUL", SEPARATOR: "tab or newline", BACKSLASH: "odd run of backslashes",
              CODE: "code", CHAR_FORM: "CHAR value", EMPTY_ROW: "one column"}


def sx(b: int) -> int:
    """signed-char extension of a byte"""
    return b - 256 if b >= 128 else b


def text_rule(s: bytes) -> int:
    """0 when the row reader gives s back as one unchanged field (oracle next_row / next_column), else the rule it breaks."""
    if not s or 0 in s:
        return ENTRY
    run = 0
    for ch in s:
        if ch in (9, 10) and run % 2 == 0:  # a separator not escaped by an odd run of backslashes
            return SEPARATOR
        run = run + 1 if ch == 0x5C else 0
    return BACKSLASH if run % 2 else 0


def writable(s: bytes) -> bool:
    return text_rule(s) == 0


def entry_rule(d: bytes, eo: list, c: int) -> int:
    """The rule entry c of the dictionary (d, eo) breaks, 0 if none; the offsets are checked before any byte is read."""
    a, b = eo[c], eo[c + 1]
    if not (a < b <= len(d)):
        return OFFSETS
    if d[b - 1] != 0:
        return ENTRY
    return text_rule(d[a:b - 1])


def char_rule(v: int) -> int:
    if v == 0:
        return 0
    if -128 <= v <= 127:
        return CHAR_FORM if v in (9, 10, 0x5C) else 0
    k, low = divmod(v - 0x5C, 256)
    return 0 if low == 0 and -128 <= k <= 127 and k != 0 else CHAR_FORM


def cell_rule(t: int, v: int, dd) -> int:
    """dd: (dict bytes, entry offsets) of a text-like column"""
    if t in TEXT_LIKE:
        if v == -1:
            return 0
        if v < -1 or v >= len(dd[1]) - 1:
            return CODE
        return entry_rule(dd[0], dd[1], v)
    if t == CHAR:
        return char_rule(v)
    return 0


def cell_text(t: int, v: int, dd) -> bytes:
    if t in TEXT_LIKE:
        if v == -1:
            return b""
        return dd[0][dd[1][v]:dd[1][v + 1] - 1]
    if t == CHAR:
        if v == 0:
            return b""
        b0 = v & 0xFF
        return bytes([b0, (v >> 8) & 0xFF]) if b0 == 0x5C else bytes([b0])
    if t in UNSIGNED:
        return str(v & ((1 << 64) - 1)).encode()
    return str(v).encode()


def check(types, cols, dicts):
    """(column, row, rule) of the lowest cell at fault, or None.  cols: per column a list of int64 cells; dicts: per
    column (dict bytes, entry offsets) for text-like columns, None for the others."""
    for k, t in enumerate(types):
        if t not in KNOWN:
            return (k, None, None)
    for k, t in enumerate(types):
        for r, v in enumerate(cols[k]):
            rule = cell_rule(t, v, dicts[k])
            if not rule and len(types) == 1 and cell_text(t, v, dicts[k]) == b"":
                rule = EMPTY_ROW
            if rule:
                return (k, r, rule)
    return None


def render(types, cols, dicts) -> bytes:
    """The rows zdwb_render_columns writes for a table that passes check()."""
    texts = [[cell_text(t, v, dicts[k]) for v in cols[k]] for k, t in enumerate(types)]
    return b"".join(b"\t".join(row) + b"\n" for row in zip(*texts))


def make_dict(ents) -> tuple:
    """(dict bytes, entry offsets) laid out as a block's dictionary: origin NUL, then every entry NUL-terminated."""
    d = b"\0" + b"".join(e + b"\0" for e in ents)
    eo, at = [], 1
    for e in ents:
        eo.append(at)
        at += len(e) + 1
    eo.append(at)
    return d, eo
