"""Python restatement of zdwb_parse_numbers and zdwb_format_numbers (include/zdw_b200.h), the oracle of
tests/test_gpu_numbers.py.  It is held to datetime and decimal.Decimal in tests/test_numbers_host.py."""
from __future__ import annotations

DATETIME, DECIMAL = 0, 1  # ZDWB_NUM_*
INT64_MIN, INT64_MAX = -(1 << 63), (1 << 63) - 1
US_PER_DAY = 86_400_000_000
DT_MIN = -62_135_596_800_000_000          # 0001-01-01 00:00:00
DT_MAX = 253_402_300_800_000_000 - 1      # 9999-12-31 23:59:59.999999
DIGITS = frozenset(b"0123456789")


def days_from_civil(y: int, m: int, d: int) -> int:
    """days from 1970-01-01 to y-m-d, proleptic Gregorian"""
    y -= m <= 2
    era = y // 400
    yoe = y - era * 400
    doy = (153 * (m - 3 if m > 2 else m + 9) + 2) // 5 + d - 1
    doe = yoe * 365 + yoe // 4 - yoe // 100 + doy
    return era * 146097 + doe - 719468


def civil_from_days(z: int) -> tuple[int, int, int]:
    z += 719468
    era = z // 146097
    doe = z - era * 146097
    yoe = (doe - doe // 1460 + doe // 36524 - doe // 146096) // 365
    doy = doe - (365 * yoe + yoe // 4 - yoe // 100)
    mp = (5 * doy + 2) // 153
    d = doy - (153 * mp + 2) // 5 + 1
    m = mp + 3 if mp < 10 else mp - 9
    return yoe + era * 400 + (m <= 2), m, d


def _leap(y: int) -> bool:
    return y % 4 == 0 and (y % 100 != 0 or y % 400 == 0)


def _num(s: bytes) -> int | None:
    return int(s) if s and all(c in DIGITS for c in s) else None


def parse_datetime(s: bytes) -> int | None:
    """microseconds since 1970-01-01 of "YYYY-MM-DD[ HH:MM:SS[.F{1,6}]]", None when s is not one or names no real time"""
    L = len(s)
    if L not in (10, 19) and not 21 <= L <= 26:
        return None
    if s[4:5] != b"-" or s[7:8] != b"-":
        return None
    y, mo, d = _num(s[0:4]), _num(s[5:7]), _num(s[8:10])
    h = mi = sec = us = 0
    if L > 10:
        if s[10:11] != b" " or s[13:14] != b":" or s[16:17] != b":":
            return None
        h, mi, sec = _num(s[11:13]), _num(s[14:16]), _num(s[17:19])
    if L > 19:
        if s[19:20] != b".":
            return None
        f = _num(s[20:])
        us = None if f is None else f * 10 ** (26 - L)
    if None in (y, mo, d, h, mi, sec, us):
        return None
    if y == 0 or not 1 <= mo <= 12 or h > 23 or mi > 59 or sec > 59:
        return None
    mdays = [31, 29 if _leap(y) else 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31][mo - 1]
    if not 1 <= d <= mdays:
        return None
    return days_from_civil(y, mo, d) * US_PER_DAY + ((h * 60 + mi) * 60 + sec) * 1_000_000 + us


def parse_decimal(s: bytes, scale: int) -> int | None:
    """[+-]?(D+(.D*)?|.D+) times 10^scale, None when s is not one, is not exact at the scale or leaves int64"""
    neg = s[:1] == b"-"
    body = s[1:] if s[:1] in (b"+", b"-") else s
    ip, dot, fp = body.partition(b".")
    if not (ip or fp) or any(c not in DIGITS for c in ip + fp):
        return None
    if any(c != 0x30 for c in fp[scale:]):
        return None
    m = int(ip or b"0") * 10 ** scale + int(fp[:scale].ljust(scale, b"0") or b"0")
    v = -m if neg else m
    return v if INT64_MIN <= v <= INT64_MAX else None


def parse(s: bytes, kind: int, digits: int = 0) -> tuple[int, bool]:
    """(value, ok) as zdwb_parse_numbers gives them: (0, False) for a text it refuses"""
    v = parse_datetime(s) if kind == DATETIME else parse_decimal(s, digits)
    return (0, False) if v is None else (v, True)


def format_datetime(us: int, digits: int) -> bytes:
    days, rem = divmod(us, US_PER_DAY)
    y, m, d = civil_from_days(days)
    sec, frac = divmod(rem, 1_000_000)
    t = b"%04d-%02d-%02d %02d:%02d:%02d" % (y, m, d, sec // 3600, sec // 60 % 60, sec % 60)
    return t + (b".%06d" % frac)[:digits + 1] if digits else t


def format_decimal(v: int, scale: int) -> bytes:
    ip, fp = divmod(abs(v), 10 ** scale)
    t = (b"-" if v < 0 else b"") + str(ip).encode()
    return t + b"." + str(fp).zfill(scale).encode() if scale else t


def format_text(v: int, kind: int, digits: int) -> bytes:
    return format_datetime(v, digits) if kind == DATETIME else format_decimal(v, digits)


def format_error(values: list, kind: int, digits: int):
    """(index, why) of the lowest value zdwb_format_numbers refuses, why in "order", "range", "multiple"; None if none"""
    for i, v in enumerate(values):
        if i and values[i - 1] >= v:
            return i, "order"
        if kind == DATETIME:
            if not DT_MIN <= v <= DT_MAX:
                return i, "range"
            if v % 10 ** (6 - digits):
                return i, "multiple"
    return None


def format_numbers(values: list, kind: int, digits: int) -> tuple[list, list]:
    """(entries sorted bytewise, codes): codes[i] is the index of values[i]'s text among the entries"""
    texts = [format_text(v, kind, digits) for v in values]
    ents = sorted(texts)
    where = {t: j for j, t in enumerate(ents)}
    return ents, [where[t] for t in texts]
