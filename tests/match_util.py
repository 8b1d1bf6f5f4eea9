"""Python restatement of zdwb_match_like and zdwb_find_strings (include/zdw_b200.h), the oracle of the GPU tests.  It is
held to sqlite's LIKE and to bisect in tests/test_match_host.py."""
from __future__ import annotations


def _fold(c: int, ignore_case: bool) -> int:
    return c + 32 if ignore_case and 0x41 <= c <= 0x5A else c


def compile_like(pattern: bytes, escape: int | None = 0x5C, ignore_case: bool = False):
    """The pattern as a list of segments split at the unescaped '%'; each segment a list of bytes (folded under
    ignore_case) and None for '_'.  ValueError for a pattern that ends in a lone escape byte."""
    segs, cur, i = [], [], 0
    while i < len(pattern):
        c = pattern[i]
        if escape is not None and c == escape:
            i += 1
            if i == len(pattern):
                raise ValueError("the pattern ends in a lone escape byte")
            cur.append(_fold(pattern[i], ignore_case))
        elif c == 0x25:  # '%'
            segs.append(cur)
            cur = []
        elif c == 0x5F:  # '_'
            cur.append(None)
        else:
            cur.append(_fold(c, ignore_case))
        i += 1
    segs.append(cur)
    return segs


def like(s: bytes, pattern: bytes, escape: int | None = 0x5C, ignore_case: bool = False) -> bool:
    """SQL LIKE over the whole of s, bytewise: '%' any run, '_' one byte, escape + byte that byte, ASCII folding."""
    segs = compile_like(pattern, escape, ignore_case)
    t = [_fold(c, ignore_case) for c in s]

    def at(seg, pos):
        return all(e is None or t[pos + j] == e for j, e in enumerate(seg))

    if len(segs) == 1:
        return len(t) == len(segs[0]) and at(segs[0], 0)
    first, last = segs[0], segs[-1]
    if len(first) + len(last) > len(t) or not at(first, 0) or not at(last, len(t) - len(last)):
        return False
    pos, end = len(first), len(t) - len(last)
    for seg in segs[1:-1]:
        while pos + len(seg) <= end and not at(seg, pos):
            pos += 1
        if pos + len(seg) > end:
            return False
        pos += len(seg)
    return True


def lower_bound(entries: list, q: bytes) -> int:
    """The number of entries bytewise less than q (entries sorted, distinct); a plain binary search."""
    lo, hi = 0, len(entries)
    while lo < hi:
        mid = (lo + hi) // 2
        if entries[mid] < q:
            lo = mid + 1
        else:
            hi = mid
    return lo


def dict_bytes(ents: list) -> tuple[bytes, list]:
    """A dictionary laid out as a block's: the origin NUL, then every entry NUL-terminated; and its entry offsets."""
    d = b"\0" + b"".join(e + b"\0" for e in ents)
    eo, at = [], 1
    for e in ents:
        eo.append(at)
        at += len(e) + 1
    eo.append(at)
    return d, eo
