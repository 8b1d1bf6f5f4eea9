"""GPU tests of numbers from and to text (zdwb_parse_numbers, zdwb_format_numbers) and of zdw_b200.numbers (to_datetime,
to_decimal, from_datetime, from_decimal).  The oracles are the Python restatement in tests/numbers_util.py (itself held to
datetime and decimal.Decimal by tests/test_numbers_host.py), the goldens' .sql text, and the C restatement of the
encoder for written files."""
import ctypes as C
import lzma
import random

import pytest

import match_util as M
import numbers_util as N
import oracle as O
from columns_util import DATETIME, DECIMAL, VARCHAR
from test_gpu_match import dev_dict
from test_numbers_host import DEC_EDGES, DT_EDGES, random_datetime_texts, random_decimal_texts, random_values

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


def check_parse(ctx, ents, kind, digits, null_text):
    import torch
    d, eo = dev_dict(ents)
    torch.cuda.synchronize()
    values, ok = ctx.parse_numbers(d, eo, kind, digits=digits, null_text=null_text)
    assert values.dtype == torch.int64 and ok.dtype == torch.bool and values.numel() == ok.numel() == len(ents) + 1
    want = [N.parse(s, kind, digits) for s in ents + [null_text]]
    assert values.cpu().tolist() == [v for v, _ in want], (kind, digits)
    assert ok.cpu().tolist() == [k for _, k in want], (kind, digits)
    return sum(k for _, k in want)


# ----------------------------------------------------------------------------- 1. parse against the restatement

@pytest.mark.parametrize("digits", [0, 6])
def test_parse_datetime_random_dictionaries(ctx, digits):
    rng = random.Random(10 + digits)
    ents = sorted(set(DT_EDGES + random_datetime_texts(rng, 20000) + [b"x" * n for n in (26, 27, 4096)]))
    assert check_parse(ctx, ents, N.DATETIME, digits, b"") > 5000
    for null in (b"", b"2018-12-31 00:01:00", b"0000-00-00 00:00:00", b"2000-02-29"):
        check_parse(ctx, ents[:100], N.DATETIME, digits, null)
    for small in ([], [b"2020-01-01"], [b"2020-01-01", b"2020-01-01 00:00:00.000001"]):
        check_parse(ctx, small, N.DATETIME, digits, b"1970-01-01")


@pytest.mark.parametrize("scale", [0, 1, 2, 12, 18])
def test_parse_decimal_random_dictionaries(ctx, scale):
    rng = random.Random(20 + scale)
    ents = sorted(set(DEC_EDGES + random_decimal_texts(rng, 20000) + [b"1" * 2000, b"0" * 3000 + b"5"]))
    assert check_parse(ctx, ents, N.DECIMAL, scale, b"0.000000000000") > 2000
    for null in (b"", b"0.000000000000", b"-1", b"1e3"):
        check_parse(ctx, ents[:100], N.DECIMAL, scale, null)
    check_parse(ctx, [], N.DECIMAL, scale, b"0.000000000000")


# ----------------------------------------------------------------------------- 2. the goldens

def sql_rows(name):
    """(first field, last field) of every row of the golden's TSV source"""
    return [(r.split(b"\t", 1)[0], r.rsplit(b"\t", 1)[1]) for r in lzma.decompress(O.golden(f"{name}.sql.xz")).split(b"\n") if r]


def test_movie_tickets():
    import torch
    from zdw_b200 import read_table, to_datetime, to_decimal
    hdr, t = read_table(O.golden("movie_tickets.zdw"))
    assert hdr.types[0] == DATETIME and hdr.types[5] == DECIMAL
    us, ok_us = to_datetime(hdr, t, 0)
    cents, ok_c = to_decimal(hdr, t, 5, scale=2)
    rows = sql_rows("movie_tickets")
    assert len(rows) == us.numel() == cents.numel()
    want_us = [N.parse(r[0], N.DATETIME) for r in rows]
    want_c = [N.parse(r[1], N.DECIMAL, 2) for r in rows]
    assert all(k for _, k in want_us) and all(k for _, k in want_c)
    assert us.cpu().tolist() == [v for v, _ in want_us] and bool(ok_us.all())
    assert cents.cpu().tolist() == [v for v, _ in want_c] and bool(ok_c.all())
    # revenue per day, in torch, against the host's sums
    day = us // N.US_PER_DAY
    days, inv = torch.unique(day, return_inverse=True)
    per_day = torch.zeros(days.numel(), dtype=torch.int64, device=day.device).index_add_(0, inv, cents)
    host = {}
    for (u, _), (c, _) in zip(want_us, want_c):
        host[u // N.US_PER_DAY] = host.get(u // N.US_PER_DAY, 0) + c
    assert dict(zip(days.cpu().tolist(), per_day.cpu().tolist())) == host
    # at scale 1 the cells with two fraction digits are not exact
    _, ok1 = to_decimal(hdr, t, 5, scale=1)
    want1 = [N.parse(r[1], N.DECIMAL, 1) for r in rows]
    assert ok1.cpu().tolist() == [k for _, k in want1] and 0 < sum(k for _, k in want1) < len(rows)
    with pytest.raises(ValueError):  # movie_rank is a number column
        to_decimal(hdr, t, 2, scale=0)


def test_analytics_hits_and_null_cells():
    from zdw_b200 import ColumnTable, read_table, to_datetime, to_decimal
    hdr, t = read_table(O.golden("analytics-hits.zdw"))
    k_dec = t.columns.index(hdr.names.index("decimal52"))
    k_dt = t.columns.index(hdr.names.index("datetime6"))
    v, ok = to_decimal(hdr, t, k_dec, scale=12)
    assert v.cpu().tolist() == [10 ** 12] * v.numel() and bool(ok.all())
    us, ok_us = to_datetime(hdr, t, k_dt)
    want = [N.parse(s or b"", N.DATETIME) for s in t.strings(k_dt)]
    assert us.cpu().tolist() == [w for w, _ in want] and ok_us.cpu().tolist() == [k for _, k in want]
    # code -1: 0 and valid on a DECIMAL column ("0.000000000000"), invalid on the others ("")
    values = t.values.clone()
    values[k_dec, ::7] = -1
    values[k_dt, ::5] = -1
    t2 = ColumnTable(values, t.dicts, t.columns, t.block_rows)
    v2, ok2 = to_decimal(hdr, t2, k_dec, scale=12)
    assert v2.cpu().tolist() == [0 if i % 7 == 0 else 10 ** 12 for i in range(v2.numel())] and bool(ok2.all())
    us2, ok_us2 = to_datetime(hdr, t2, k_dt)
    assert ok_us2.cpu().tolist() == [i % 5 != 0 and want[i][1] for i in range(us2.numel())]
    assert us2.cpu().tolist() == [0 if i % 5 == 0 else want[i][0] for i in range(us2.numel())]
    k_txt = next(k for k, c in enumerate(t.columns) if hdr.types[c] == VARCHAR)
    values[k_txt, ::3] = -1
    d3, ok3 = to_decimal(hdr, ColumnTable(values, t.dicts, t.columns, t.block_rows), k_txt, scale=0)
    assert not any(ok3.cpu().tolist()[::3]) and all(x == 0 for x in d3.cpu().tolist()[::3])


# ----------------------------------------------------------------------------- 3. format against the restatement

def check_format(ctx, vals, kind, digits):
    import torch
    v = torch.tensor(vals, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    m = ctx.format_numbers(v, kind, digits=digits)
    ents, codes = N.format_numbers(vals, kind, digits)
    d, eo = M.dict_bytes(ents) if ents else (b"", [0])
    assert bytes(m.dict.cpu().numpy().tobytes()) == d
    assert m.entry_off.cpu().tolist() == eo
    assert m.codes.cpu().tolist() == codes
    if kind == N.DATETIME:
        assert codes == list(range(len(vals)))
    if ents:  # dense and strictly increasing: every entry finds itself
        rank, found = ctx.find_strings(m.dict, m.entry_off, ents)
        assert rank.cpu().tolist() == list(range(len(ents))) and bool(found.all())
        values, ok = ctx.parse_numbers(m.dict, m.entry_off, kind, digits=digits)
        assert bool(ok[:-1].all()) and values[m.codes].cpu().tolist() == vals
    return m


@pytest.mark.parametrize("kind,digits", [(0, 0), (0, 3), (0, 6), (1, 0), (1, 2), (1, 12), (1, 18)])
def test_format_random_values(ctx, kind, digits):
    rng = random.Random(30 + 10 * kind + digits)
    for n in (0, 1, 2, 1000, 70000, 300000):  # 70000 and more: the radix path of the string sort
        vals = random_values(rng, kind, digits, n)[:n] if n else []
        check_format(ctx, vals, kind, digits)


# ----------------------------------------------------------------------------- 4. round trip through a file

def test_round_trip_through_write_table(ctx, tmp_path):
    import torch
    from zdw_b200 import ColumnTable, FileHeader, from_datetime, from_decimal, read_table, to_datetime, to_decimal
    from test_gpu_write import oracle_file, written
    rng = random.Random(40)
    n = 5000
    dev = "cuda"
    us = torch.tensor([rng.randrange(N.DT_MIN // 1000, N.DT_MAX // 1000) * 1000 for _ in range(n)], dtype=torch.int64, device=dev)
    us[::4] = us[1::4][:us[::4].numel()]  # repeated values
    cents = torch.tensor([rng.randrange(N.INT64_MIN, N.INT64_MAX + 1) >> rng.randrange(64) for _ in range(n)], dtype=torch.int64,
                         device=dev)
    cents[::5] = 0
    cents[1] = N.INT64_MIN
    valid_us = torch.tensor([rng.random() < 0.9 for _ in range(n)], device=dev)
    valid_c = torch.tensor([rng.random() < 0.9 for _ in range(n)], device=dev)
    c_us, d_us = from_datetime(us, valid_us, frac_digits=3)
    c_c, d_c = from_decimal(cents, valid_c, scale=2)
    c_i, d_i = from_decimal(cents, scale=0)  # a VARCHAR column of integers
    assert c_us[~valid_us].eq(-1).all() and c_c[~valid_c].eq(-1).all() and c_i.ge(0).all()
    hdr = FileHeader(11, {}, ["when", "amount", "count"], [DATETIME, DECIMAL, VARCHAR], [0, 0, 32], 0)
    t = ColumnTable(torch.stack([c_us, c_c, c_i]), [d_us, d_c, d_i], [0, 1, 2], [n // 2, n - n // 2])
    got = written(tmp_path, hdr, t)
    assert got == oracle_file(hdr, t, t.block_rows)
    h2, back = read_table(got)
    u2, ok_u = to_datetime(h2, back, 0)
    c2, ok_c = to_decimal(h2, back, 1, scale=2)
    i2, ok_i = to_decimal(h2, back, 2, scale=0)
    assert ok_u.tolist() == valid_us.tolist() and u2.tolist() == torch.where(valid_us, us, 0).tolist()
    assert bool(ok_c.all()) and c2.tolist() == torch.where(valid_c, cents, 0).tolist()  # an empty DECIMAL reads as 0
    assert bool(ok_i.all()) and i2.tolist() == cents.tolist()
    for k in range(3):  # the written dictionaries are the formatted ones, less the entries of no row
        assert sorted(set(back.strings(k)) - {None}) == sorted(set(t.strings(k)) - {None})


# ----------------------------------------------------------------------------- 5. errors

def test_errors_and_recovery(ctx):
    import torch
    from zdw_b200 import ZdwError, capi
    good = [b"1.5", b"2", b"x"]
    d, eo = dev_dict(good)

    def normal():
        check_parse(ctx, good, N.DECIMAL, 1, b"")
        check_format(ctx, [-5, 0, 7], N.DECIMAL, 1)

    def fails(call, code, *texts):
        torch.cuda.synchronize()
        with pytest.raises(ZdwError) as ei:
            call()
        assert ei.value.code == code, ei.value
        assert all(x in ei.value.msg for x in texts), ei.value.msg
        normal()  # the context works normally at its next call

    L = ctx._L
    part = capi._CodePart(d.data_ptr(), eo.data_ptr(), 3, d.numel(), None, 0)
    opts = capi._NumberOpts(1, 2, b"", 0)
    po, mo = capi._ParseOut(), capi._MergeOut()
    vals = torch.tensor([1, 2, 3], dtype=torch.int64, device="cuda")
    # NULL arguments
    assert L.zdwb_parse_numbers(ctx._h, None, C.byref(opts), C.byref(po)) == 4
    assert L.zdwb_parse_numbers(ctx._h, C.byref(part), None, C.byref(po)) == 4
    assert L.zdwb_parse_numbers(ctx._h, C.byref(part), C.byref(opts), None) == 4
    assert L.zdwb_format_numbers(ctx._h, C.c_void_p(vals.data_ptr()), 3, None, C.byref(mo)) == 4
    assert L.zdwb_format_numbers(ctx._h, C.c_void_p(vals.data_ptr()), 3, C.byref(opts), None) == 4
    assert L.zdwb_format_numbers(ctx._h, None, 3, C.byref(opts), C.byref(mo)) == 4
    assert "NULL values" in ctx.last_error()
    for bad in (capi._CodePart(None, eo.data_ptr(), 3, d.numel(), None, 0), capi._CodePart(d.data_ptr(), None, 3, d.numel(), None, 0)):
        assert L.zdwb_parse_numbers(ctx._h, C.byref(bad), C.byref(opts), C.byref(po)) == 4
    assert L.zdwb_parse_numbers(ctx._h, C.byref(part), C.byref(capi._NumberOpts(1, 0, None, 3)), C.byref(po)) == 4
    assert "null_text" in ctx.last_error()
    normal()
    # kind and digits
    for kind, digits, fmt in ((2, 0, False), (-1, 0, True), (1, 19, False), (1, -1, True), (0, 7, True), (0, -1, True)):
        o = capi._NumberOpts(kind, digits, None, 0)
        rc = (L.zdwb_format_numbers(ctx._h, C.c_void_p(vals.data_ptr()), 3, C.byref(o), C.byref(mo)) if fmt else
              L.zdwb_parse_numbers(ctx._h, C.byref(part), C.byref(o), C.byref(po)))
        assert rc == 4 and ("kind" in ctx.last_error() or "digits" in ctx.last_error()), (kind, digits, ctx.last_error())
        normal()
    check_parse(ctx, [b"2020-01-01"], N.DATETIME, 99, b"")  # DATETIME parse ignores digits
    # entry offsets, garbage included: the lowest entry at fault is named
    for offs, low in (([1, 5, 5, 7], 1), ([1, 5, 99, 7], 1), ([1, 5, 3, 7], 1), ([1, 5, 7, 10], 2), ([9, 5, 7, 9], 0),
                      ([1 << 62, 1 << 63, 3, 2], 0), ([1, 5, 7, (1 << 64) - 1], 2)):
        bad = torch.tensor([o - (1 << 64) if o >= 1 << 63 else o for o in offs], dtype=torch.int64, device="cuda")
        for kind in (N.DATETIME, N.DECIMAL):
            fails(lambda: ctx.parse_numbers(d, bad, kind, digits=1), 4, f"entry {low} has offsets")
    # format: order, range, exactness; the lowest value is named
    for vals_, kind, digits, low, text in (
            ([1, 1], N.DECIMAL, 0, 1, "not greater"), ([5, 3, 1, 0], N.DECIMAL, 2, 1, "not greater"),
            ([0, 1, 2, 2, 1], N.DECIMAL, 0, 3, "not greater"), ([N.INT64_MAX, N.INT64_MIN], N.DECIMAL, 18, 1, "not greater"),
            ([N.DT_MIN - 1, 0], N.DATETIME, 6, 0, "outside"), ([0, N.DT_MAX + 1], N.DATETIME, 6, 1, "outside"),
            ([0, N.INT64_MAX], N.DATETIME, 0, 1, "outside"), ([N.INT64_MIN, 0], N.DATETIME, 0, 0, "outside"),
            ([0, 1_000_000, 1_000_001], N.DATETIME, 0, 2, "multiple of 10^6"), ([0, 100, 110], N.DATETIME, 4, 2, "multiple of 10^2"),
            ([-1, 5], N.DATETIME, 5, 0, "multiple of 10^1"), ([0, 10, 5], N.DATETIME, 6, 2, "not greater")):
        assert N.format_error(vals_, kind, digits)[0] == low
        vt = torch.tensor(vals_, dtype=torch.int64, device="cuda")
        fails(lambda: ctx.format_numbers(vt, kind, digits=digits), 4, f"value {low} ", text)
    # 2^32 bytes of text and more: the widest DATETIME text takes 27 bytes with its NUL
    n = -(-(1 << 32) // 27)
    big = torch.arange(n, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    fails(lambda: ctx.format_numbers(big, N.DATETIME, digits=6), 5, "2^32")
    del big
    assert L.zdwb_format_numbers(ctx._h, C.c_void_p(vals.data_ptr()), 1 << 32, C.byref(opts), C.byref(mo)) == 5
    normal()
    with pytest.raises(ValueError):
        ctx.format_numbers(torch.tensor([1.0], device="cuda"), N.DECIMAL)
