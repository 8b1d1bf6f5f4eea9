"""The TSV text of a zdwb_decode_columns cell, as the row decoder prints it (include/zdw_b200.h), for the columnar tests
and tools/columns_timing.py."""
from __future__ import annotations

# column type ids (include/zdw_b200.h, zdw_column_type_constants.h:17-35)
VARCHAR, TEXT, DATETIME, CHAR_2, CHAR = 0, 1, 2, 3, 6
TINY, SHORT, LONG, LONGLONG = 7, 8, 9, 10
DECIMAL = 11
TINYTEXT, MEDIUMTEXT, LONGTEXT = 16, 17, 18
TEXT_LIKE = {VARCHAR, TEXT, DATETIME, CHAR_2, DECIMAL, TINYTEXT, MEDIUMTEXT, LONGTEXT}
UNSIGNED = {TINY, SHORT, LONG, LONGLONG}

INT64_MIN = -(1 << 63)
# lltoa's text of INT64_MIN: every remainder is negative, the digit byte is 0x30 - d (SURVEY App. B-22)
INT64_MIN_TEXT = b"-" + bytes(0x30 - int(ch) for ch in "9223372036854775808")


def entries(dict_bytes: bytes, entry_off: list) -> list:
    """The dictionary's entries (entry i = dict[entry_off[i] : entry_off[i + 1] - 1])."""
    return [dict_bytes[a:b - 1] for a, b in zip(entry_off, entry_off[1:])]


def render(t: int, v: int, ents: list) -> bytes:
    """The text of a cell of a column of type t holding the int64 v (ents: the block's dictionary entries)."""
    if t in TEXT_LIKE:
        if v == -1:
            return b"0.000000000000" if t == DECIMAL else b""
        return ents[v]
    if t == CHAR:
        b0 = v & 0xFF
        if b0 == 0:
            return b""
        return bytes([b0, (v >> 8) & 0xFF]) if b0 == ord("\\") else bytes([b0])
    if t in UNSIGNED:
        return str(v & ((1 << 64) - 1)).encode()
    return INT64_MIN_TEXT if v == INT64_MIN else str(v).encode()
