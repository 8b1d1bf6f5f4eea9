"""Numbers from and to text, the parts that need no GPU: the ctypes mirrors of the new structs against a C compiler's
layout, the exports, and the Python restatement of parse and format (tests/numbers_util.py, the oracle of
tests/test_gpu_numbers.py) against independent oracles: datetime.datetime with a strict regex for DATETIME and
decimal.Decimal for DECIMAL."""
import ctypes as C
import datetime as dt
import decimal
import random
import re
import subprocess

import pytest

import numbers_util as N
from test_abi import HEADER

EPOCH = dt.datetime(1970, 1, 1)
DT_RE = re.compile(rb"([0-9]{4})-([0-9]{2})-([0-9]{2})(?: ([0-9]{2}):([0-9]{2}):([0-9]{2})(?:\.([0-9]{1,6}))?)?")
DEC_RE = re.compile(rb"[+-]?(?:[0-9]+(?:\.[0-9]*)?|\.[0-9]+)")


def test_number_structs_match_the_header_layout(tmp_path):
    from zdw_b200 import capi
    pairs = [("zdwb_number_opts", capi._NumberOpts), ("zdwb_parse_out", capi._ParseOut)]
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    lines = ['#include <stddef.h>', '#include <stdio.h>', f'#include "{HEADER}"', "int main(void) {"]
    fields = {}
    for cname, _ in pairs:
        body = re.search(r"typedef struct\s*\{([^}]*)\}\s*" + cname + r"\s*;", text).group(1)
        fields[cname] = re.findall(r"([A-Za-z_][A-Za-z0-9_]*)\s*(?:\[[^\]]*\])?\s*;", body)
        lines.append(f'  printf("{cname} %zu", sizeof({cname}));')
        for f in fields[cname]:
            lines.append(f'  printf(" %zu", offsetof({cname}, {f}));')
        lines.append('  printf("\\n");')
    lines += ['  printf("%d %d\\n", ZDWB_NUM_DATETIME, ZDWB_NUM_DECIMAL);', "  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    for (cname, mirror), line in zip(pairs, out):
        nums = [int(x) for x in line.split()[1:]]
        assert C.sizeof(mirror) == nums[0], cname
        assert [f[0] for f in mirror._fields_] == fields[cname]
        assert [getattr(mirror, f[0]).offset for f in mirror._fields_] == nums[1:], cname
    assert out[-1].split() == [str(capi.NUM_DATETIME), str(capi.NUM_DECIMAL)] == [str(N.DATETIME), str(N.DECIMAL)]


def test_library_exports_the_number_calls_at_abi_5():
    from zdw_b200 import capi
    lib = C.CDLL(str(capi.lib_path()))
    for name in ("zdwb_parse_numbers", "zdwb_format_numbers"):
        assert hasattr(lib, name)
        assert name in capi.EXPORTED_SYMBOLS
        assert re.search(rf"\bint {name}\(", HEADER.read_text())
    assert capi.load_library().zdwb_abi_version() == 5


# ----------------------------------------------------------------------------- the independent oracles

def oracle_datetime(s: bytes):
    m = DT_RE.fullmatch(s)
    if not m:
        return None
    y, mo, d, h, mi, sec, f = m.groups()
    try:
        t = dt.datetime(int(y), int(mo), int(d), int(h or 0), int(mi or 0), int(sec or 0), int((f or b"0").ljust(6, b"0")))
    except ValueError:
        return None
    return (t - EPOCH) // dt.timedelta(microseconds=1)


def oracle_decimal(s: bytes, scale: int):
    if not DEC_RE.fullmatch(s):
        return None
    with decimal.localcontext() as c:
        c.prec = 200
        q = decimal.Decimal(s.decode()).scaleb(scale)
        if q != q.to_integral_value():
            return None
        v = int(q)
    return v if N.INT64_MIN <= v <= N.INT64_MAX else None


DT_EDGES = [
    b"2000-02-29", b"2000-02-29 12:00:00", b"1900-02-29", b"1900-02-28 23:59:59", b"2004-02-29", b"2100-02-29",
    b"2400-02-29 00:00:00", b"0000-00-00 00:00:00", b"0000-00-00", b"0001-01-01 00:00:00", b"9999-12-31 23:59:59.999999",
    b"1970-01-01 00:00:00", b"1969-12-31 23:59:59.999999", b"2018-12-31 24:00:00", b"2018-12-31 23:60:00",
    b"2018-12-31 23:59:60", b"2018-13-01", b"2018-00-10", b"2018-04-31", b"2018-04-30", b"2018-01-00",
    b"2018-12-31 00:01:00.", b"2018-12-31 00:01:00.1", b"2018-12-31 00:01:00.12", b"2018-12-31 00:01:00.123",
    b"2018-12-31 00:01:00.1234", b"2018-12-31 00:01:00.12345", b"2018-12-31 00:01:00.123456",
    b"2018-12-31 00:01:00.1234567", b" 2018-12-31 00:01:00", b"2018-12-31 00:01:00 ", b"2018-12-31 ", b" 2018-12-31",
    b"2018-12-31T00:01:00", b"2018-12-31 00:01", b"2018/12/31", b"18-12-31", b"+018-12-31", b"2018-1-31", b"2018-12-31\n",
    b"", b"0", b"2018-12-31 00:01:00.12a", b"2018-12-31 0a:01:00", b"\xd9\xa2018-12-31", b"2018-12-31 00:01:00.-1",
    b"2018-12-31 00:01:00" + b"0" * 200,
]

DEC_EDGES = [
    b"+4", b"-0", b"+0", b"0", b".5", b"5.", b"-.5", b"+5.", b"-", b"+", b".", b"-.", b"1e3", b"1E3", b"1.5e1", b" 1",
    b"1 ", b"1,5", b"1..5", b"1.5.", b"--1", b"+-1", b"0x10", b"1.50", b"1.05", b"1.000000000000", b"0.000000000000",
    b"0" * 40 + b"1", b"-" + b"0" * 40 + b"7.25", b"1." + b"0" * 40, b"9223372036854775807", b"-9223372036854775808",
    b"9223372036854775808", b"-9223372036854775809", b"18446744073709551616", b"99999999999999999999999",
    b"0" * 40 + b"9223372036854775807", b"9.223372036854775807", b"-9.223372036854775808", b"9.223372036854775808",
    b"0.000000000000000001", b"0.0000000000000000001", b"0.0000000000000000010", b"1370.25", b"1392.0", b"",
    b"\xd9\xa1", b"1\x00",
]


def random_datetime_texts(rng, n):
    out = []
    for _ in range(n):
        v = rng.randrange(N.DT_MIN, N.DT_MAX + 1)
        nd = rng.choice([0, 0, 1, 2, 3, 4, 5, 6])
        s = N.format_datetime(v, nd) if rng.random() < 0.8 else N.format_datetime(v, 0)[:10]
        r = rng.random()
        if r < 0.3:  # a random byte changed, cut or added
            i = rng.randrange(len(s))
            s = s[:i] + bytes([rng.choice(b"0123456789 -:.9x\x00")]) + s[i + 1:]
        elif r < 0.35:
            s = s[:rng.randrange(len(s))]
        elif r < 0.4:
            s += bytes([rng.choice(b"0 .")])
        elif r < 0.5:  # day, hour, minute or second past its end
            s = s[:8] + rng.choice([b"29", b"30", b"31", b"32"]) + s[10:] if len(s) >= 10 else s
        out.append(s)
    return out


def random_decimal_texts(rng, n):
    out = []
    for _ in range(n):
        ip = "".join(rng.choice("0123456789") for _ in range(rng.choice([0, 1, 2, 5, 12, 18, 19, 20, 25])))
        fp = "".join(rng.choice("0000123456789") for _ in range(rng.choice([0, 0, 1, 2, 3, 12, 18, 20])))
        s = rng.choice(["", "", "-", "+"]) + ip + (rng.choice([".", ""]) if not fp else "." + fp)
        if rng.random() < 0.1:
            i = rng.randrange(len(s) + 1)
            s = s[:i] + rng.choice(".e-+ 0a") + s[i:]
        out.append(s.encode())
    return out


def test_datetime_restatement_agrees_with_datetime():
    rng = random.Random(1)
    texts = DT_EDGES + random_datetime_texts(rng, 30000)
    ok = 0
    for s in texts:
        want = oracle_datetime(s)
        assert N.parse_datetime(s) == want, s
        assert N.parse(s, N.DATETIME, rng.randint(0, 18)) == ((0, False) if want is None else (want, True))
        ok += want is not None
    assert 10000 < ok < len(texts) - 5000
    assert N.parse_datetime(b"2000-02-29") is not None and N.parse_datetime(b"1900-02-29") is None
    assert N.parse_datetime(b"0000-00-00 00:00:00") is None and N.parse_datetime(b"2018-12-31 24:00:00") is None
    assert N.parse_datetime(b"1970-01-01") == 0 and N.parse_datetime(b"1969-12-31 23:59:59.999999") == -1
    assert N.parse_datetime(b"0001-01-01 00:00:00") == N.DT_MIN and N.parse_datetime(b"9999-12-31 23:59:59.999999") == N.DT_MAX
    assert N.parse_datetime(b"2018-12-31 00:01:00.5") == N.parse_datetime(b"2018-12-31 00:01:00.500000")


@pytest.mark.parametrize("scale", [0, 1, 2, 6, 12, 18])
def test_decimal_restatement_agrees_with_decimal(scale):
    rng = random.Random(scale)
    texts = DEC_EDGES + random_decimal_texts(rng, 20000)
    ok = 0
    for s in texts:
        want = oracle_decimal(s, scale)
        assert N.parse_decimal(s, scale) == want, (s, scale)
        ok += want is not None
    assert 2000 < ok < len(texts) - 2000


def test_decimal_edges():
    P = N.parse_decimal
    assert P(b"+4", 0) == 4 and P(b"-0", 0) == 0 and P(b".5", 1) == 5 and P(b"5.", 0) == 5
    assert P(b"-", 0) is None and P(b".", 0) is None and P(b"1e3", 0) is None
    assert P(b"1.50", 1) == 15 and P(b"1.50", 0) is None and P(b"1.5", 2) == 150
    assert P(b"0" * 40 + b"1", 0) == 1 and P(b"0" * 40 + b"1", 18) == 10 ** 18
    assert P(b"9223372036854775807", 0) == N.INT64_MAX and P(b"9223372036854775808", 0) is None
    assert P(b"-9223372036854775808", 0) == N.INT64_MIN and P(b"-9223372036854775809", 0) is None
    assert P(b"-9.223372036854775808", 18) == N.INT64_MIN and P(b"9.223372036854775808", 18) is None
    assert P(b"1.000000000000", 12) == 10 ** 12 and P(b"0.000000000000", 12) == 0
    assert P(b"9.223372036854775807" + b"0" * 30, 18) == N.INT64_MAX


def random_values(rng, kind, digits, n):
    if kind == N.DATETIME:
        step = 10 ** (6 - digits)
        vals = {rng.randrange(N.DT_MIN // step, N.DT_MAX // step + 1) * step for _ in range(n)}
        vals |= {N.DT_MIN, N.DT_MAX // step * step, 0, -step}
    else:
        vals = {rng.randrange(N.INT64_MIN, N.INT64_MAX + 1) >> rng.randrange(64) for _ in range(n)}
        vals |= {N.INT64_MIN, N.INT64_MAX, 0, -1, 1, 10 ** digits, -10 ** digits, 10 ** digits - 1}
    return sorted(vals)


@pytest.mark.parametrize("kind,digits", [(0, 0), (0, 1), (0, 3), (0, 6), (1, 0), (1, 1), (1, 2), (1, 12), (1, 18)])
def test_format_round_trip_and_order(kind, digits):
    rng = random.Random(kind * 100 + digits)
    vals = random_values(rng, kind, digits, 5000)
    assert N.format_error(vals, kind, digits) is None
    ents, codes = N.format_numbers(vals, kind, digits)
    assert len(set(ents)) == len(ents) == len(vals)
    assert all(a < b for a, b in zip(ents, ents[1:]))
    for v, c in zip(vals, codes):
        s = ents[c]
        assert N.parse(s, kind, digits) == (v, True), (v, s)
        if kind == N.DATETIME:
            assert s == (EPOCH + dt.timedelta(microseconds=v)).isoformat(" ", "microseconds").encode()[:len(s)]
            assert len(s) == 19 + (digits + 1 if digits else 0)
        else:
            assert decimal.Decimal(s.decode()).scaleb(digits) == v
            body = s[1:] if v < 0 else s
            assert body[:1] != b"0" or body == b"0" or body.startswith(b"0.")
    if kind == N.DATETIME:
        assert codes == list(range(len(vals)))  # fixed width: the bytewise order is the numeric one
    assert N.format_decimal(N.INT64_MIN, 0) == b"-9223372036854775808"
    assert N.format_decimal(N.INT64_MIN, 18) == b"-9.223372036854775808"
    assert N.format_decimal(-5, 2) == b"-0.05" and N.format_decimal(0, 2) == b"0.00" and N.format_decimal(7, 0) == b"7"


def test_format_errors():
    assert N.format_error([1, 1], N.DECIMAL, 0) == (1, "order")
    assert N.format_error([3, 2, 1], N.DECIMAL, 0) == (1, "order")
    assert N.format_error([N.DT_MIN - 1, 0], N.DATETIME, 6) == (0, "range")
    assert N.format_error([0, N.DT_MAX + 1], N.DATETIME, 6) == (1, "range")
    assert N.format_error([0, 1_000_000, 1_000_001], N.DATETIME, 0) == (2, "multiple")
    assert N.format_error([0, 100], N.DATETIME, 4) is None
    assert N.format_error([0, 10], N.DATETIME, 4) == (1, "multiple")
