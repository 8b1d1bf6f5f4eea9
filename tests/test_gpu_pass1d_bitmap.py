"""The row-delta pass 1 sets the bits of a row's non-empty-column bitmap while it extracts the fields (and rebuilds the
bitmap from the fields that stay under -t): same bytes as the C restatement (or, for C4 slices, as the general pass 1)
with tiles of 8 and 32 KiB."""
import ctypes as C
import random

import pytest

import corpus
import gpuutil as G
import oracle as O

pytestmark = pytest.mark.gpu

TILES = [8192, 32768]
BS = b"\\"


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def c4(ctx):
    """C4 slices of 4 096 and 32 768 rows, with the general pass 1's file of each as the expected bytes."""
    import bench
    synth = bench.Synth()
    sch = O.parse_desc(synth.desc)
    out = []
    for rows, block in ((4096, 0), (32768, 3)):
        cap = synth.cap_for(rows)
        buf = (C.c_uint8 * cap)()
        n = synth.block_into(block, rows, C.addressof(buf), cap)
        tsv = bytes(memoryview(buf)[:n])
        ctx.set_tuning("enc_delta", 0)
        try:
            want = G.encode_file_with_product(ctx, sch, tsv)
        finally:
            ctx.set_tuning("enc_delta", -1)
        out.append((rows, sch, tsv, want))
    return out


# Changed fields of 15, 16 and 17 bytes (the longest compared straight-line, and one past it), longer texts, numbers,
# CHAR cells, empty cells and repeats; with `escapes`, escaped tabs and newlines inside texts.
SCHEMA = [("n0", "int(11)"), ("t0", "varchar(64)"), ("c0", "char(1)"), ("n1", "bigint(20)"), ("t1", "text"),
          ("t2", "varchar(255)"), ("n2", "int(11)"), ("t3", "varchar(32)")] * 6


def _value(rng, typ, escapes, trim):
    if typ.startswith(("int", "bigint")):
        return b"%d" % rng.choice([0, 7, 123456789012345, 999999999999999, 1234567890123456, 12345678901234567,
                                   rng.randrange(1 << 40)])
    if typ.startswith("char"):
        return rng.choice([b"a", b"Z", BS + b"t", b"-"])
    n = rng.choice([1, 5, 15, 16, 17, 40, 150])
    v = bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz0123456789") for _ in range(n))
    if escapes and rng.random() < 0.2:
        i = rng.randrange(n)
        v = v[:i] + rng.choice([BS + b"\t", BS + b"\n", BS + BS]) + v[i:]
    if trim and rng.random() < 0.3:
        v = v + b" " * rng.choice([1, 2, 3])  # e.g. 15 or 16 bytes of text + spaces: under 16 once trimmed
    return v


def wide_rows(nrows, seed, escapes=False, trim=False, tail=b""):
    rng = random.Random(seed)
    prev = None
    rows = []
    for _ in range(nrows):
        row = []
        for i, (_, typ) in enumerate(SCHEMA):
            r = rng.random()
            if prev is not None and r < 0.55:
                row.append(prev[i])
            elif r < 0.65:
                row.append(b" " * rng.choice([1, 2]) if trim else b"")
            else:
                row.append(_value(rng, typ, escapes, trim))
        rows.append(row)
        prev = row
    if tail:  # the last row's last field changes and ends right in front of the buffer's last byte
        rows[-1] = rows[-2][:-1] + [tail]
    return corpus.rows(rows)


def _check(ctx, sch, tsv, trim=False, plan=None):
    want = O.encode(sch, tsv, trim=trim, plan=plan)
    assert want.rc == 0
    got = G.encode_file_with_product(ctx, sch, tsv, trim=trim, plan=plan)
    assert got == want.data, G.first_diff(got, want.data)


@pytest.fixture
def forced(ctx, request):
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", request.param)
    yield ctx
    ctx.set_tuning("enc_delta", -1)
    ctx.set_tuning("enc_dtile", 0)


PARAMS = TILES
IDS = [f"tile{t}" for t in TILES]


@pytest.mark.parametrize("forced", PARAMS, ids=IDS, indirect=True)
def test_corpus(forced):
    for name, desc, tsv, opts in corpus.cases():
        if opts.get("expect_rc") or name.startswith("d2_"):
            continue
        sch = O.parse_desc(desc)
        trim = bool(opts.get("trim"))
        want = O.encode(sch, tsv, trim=trim)
        if want.rc != 0:
            continue
        got = G.encode_file_with_product(forced, sch, tsv, trim=trim)
        assert got == want.data, f"{name}: {G.first_diff(got, want.data)}"


@pytest.mark.parametrize("forced", PARAMS, ids=IDS, indirect=True)
def test_wide_rows_across_runs(forced):
    """Rows of a few hundred bytes to a few KiB: many of them straddle tile boundaries."""
    sch = O.parse_desc(corpus.desc(SCHEMA))
    _check(forced, sch, wide_rows(600, 1))
    _check(forced, sch, wide_rows(400, 2, escapes=True))


@pytest.mark.parametrize("forced", PARAMS, ids=IDS, indirect=True)
def test_trailing_spaces_trimmed(forced):
    sch = O.parse_desc(corpus.desc(SCHEMA))
    _check(forced, sch, wide_rows(400, 3, trim=True), trim=True)


@pytest.mark.parametrize("forced", PARAMS, ids=IDS, indirect=True)
@pytest.mark.parametrize("n", [15, 16, 17])
def test_changed_field_at_buffer_end(forced, n):
    """A changed text of 15 / 16 / 17 bytes closes the input: its loads run into the buffer's last word."""
    sch = O.parse_desc(corpus.desc(SCHEMA))
    _check(forced, sch, wide_rows(60, 4 + n, tail=b"q" * (n - 1) + b"z"))
    _check(forced, sch, wide_rows(3, 5 + n, tail=b"r" * n))


@pytest.mark.parametrize("forced", PARAMS, ids=IDS, indirect=True)
def test_block_cut_by_rows_and_spill(forced):
    sch = O.parse_desc(corpus.desc(SCHEMA))
    tsv = wide_rows(500, 6, escapes=True)
    for plan in ([(200, 3), (150, 1), (150, 0)], [(7, 20), (493, 0)]):
        _check(forced, sch, tsv, plan=plan)
    for rpb in (1, 77):
        want = O.encode(sch, tsv, rows_per_block=rpb).data
        got = G.encode_file_with_product(forced, sch, tsv, rows_per_block=rpb)
        assert got == want, f"rows_per_block {rpb}: {G.first_diff(got, want)}"


@pytest.mark.parametrize("forced", PARAMS, ids=IDS, indirect=True)
def test_c4_slices(forced, c4):
    for rows, sch, tsv, want in c4:
        got = G.encode_file_with_product(forced, sch, tsv)
        assert got == want, f"C4 {rows} rows: {G.first_diff(got, want)}"

