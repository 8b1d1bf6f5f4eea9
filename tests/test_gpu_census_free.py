"""The census-free row-delta pass 1 (`enc_census`): pass 1 finds each tile's reference row itself, numbers the tile's
rows from 0 and a scan makes the numbers global.  Every block it encodes must come out exactly as with the row census
(`enc_census=1`): the block bytes and every `zdwb_block_out` field, or the same error.  Where the existing tests do, the
bytes are also checked against the C restatement (`oracle.encode`)."""
import ctypes as C
import random

import pytest

import corpus
import gpuutil as G
import oracle as O

pytestmark = pytest.mark.gpu

FIELDS = ("data", "length", "nrows", "longest_line", "tsv_consumed", "rows_in_buffer", "ncols_used", "dict_entries",
          "dict_bytes", "dict_index_size")


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture()
def knobs(ctx):
    yield ctx
    for k, v in (("enc_census", -1), ("enc_delta", -1), ("enc_dtile", 0), ("ht_initial_log2", 20), ("kernel_timing", 0)):
        ctx.set_tuning(k, v)


def _encode(ctx, census, types, tsv, kernels=None, **kw):
    """(block fields, None) or (None, (code, bad_row, message)) of one encode_block call with enc_census = census;
    the kernels it launched go to `kernels` (a set)."""
    from zdw_b200 import ZdwError
    ctx.set_tuning("enc_census", census)
    ctx.set_tuning("kernel_timing", 1)
    ctx.kernel_times()
    try:
        blk = ctx.encode_block(types, tsv, **kw)
    except ZdwError as e:
        return None, (e.code, e.bad_row, ctx.last_error())
    finally:
        if kernels is not None:
            kernels.update(ctx.kernel_times())
    return {f: getattr(blk, f) for f in FIELDS}, None


def _same(ctx, types, tsv, what="", **kw):
    """Census-free (0) and census (1) encodes of one window agree; returns the census-free result.  Where the census
    run kept the row-delta path (census, no general pass 1), the census-free run must have done without the census -
    a fall-back to it would compare the census with itself."""
    k0, k1 = set(), set()
    got = _encode(ctx, 0, types, tsv, k0, **kw)
    want = _encode(ctx, 1, types, tsv, k1, **kw)
    if "k_row_census" in k1 and "k_tile_count" not in k1:
        assert "k_row_fixup" in k0 and "k_row_census" not in k0, f"{what}: census-free run launched {sorted(k0)}"
    if got != want:
        if got[0] and want[0] and got[0]["data"] != want[0]["data"]:
            raise AssertionError(f"{what}: {G.first_diff(got[0]['data'], want[0]['data'])}")
        raise AssertionError(f"{what}: census-free {got[0] and {k: v for k, v in got[0].items() if k != 'data'} or got[1]} "
                             f"!= census {want[0] and {k: v for k, v in want[0].items() if k != 'data'} or want[1]}")
    return got


def _file(ctx, census, sch, tsv, trim=False):
    ctx.set_tuning("enc_census", census)
    return G.encode_file_with_product(ctx, sch, tsv, trim=trim)


@pytest.mark.parametrize("tile", [2048, 8192, 32768])
def test_corpus_and_golden(knobs, tile):
    ctx = knobs
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", tile)
    for name, desc, tsv, opts in corpus.cases():
        sch = O.parse_desc(desc)
        trim = bool(opts.get("trim"))
        _same(ctx, sch.types, tsv, name, trim=trim)
        want = O.encode(sch, tsv, trim=trim)
        if want.rc == 0:
            got = _file(ctx, 0, sch, tsv, trim=trim)
            assert got == want.data, f"{name}: {G.first_diff(got, want.data)}"
    sch = O.parse_desc(O.golden("analytics-hits.desc.sql"))
    tsv = O.golden("analytics-hits.sql")
    _same(ctx, sch.types, tsv, "C3")
    want = O.golden_to_v11(O.golden("analytics-hits.zdw"))
    got = _file(ctx, 0, sch, tsv)
    assert got == want, G.first_diff(got, want)


def _c4_block(synth, block, rows):
    cap = synth.cap_for(rows)
    buf = (C.c_uint8 * cap)()
    n = synth.block_into(block, rows, C.addressof(buf), cap)
    return bytes(memoryview(buf)[:n])


@pytest.mark.parametrize("rows", [4096, 32768, 131072])
def test_c4_blocks_on_one_context_skip_the_census(rows):
    """Under the default knob the first block of a context takes the census and every later one does without it."""
    import bench
    from zdw_b200 import Context
    synth = bench.Synth()
    sch = O.parse_desc(synth.desc)
    blocks = [_c4_block(synth, b, rows) for b in range(3)]
    with Context(0) as ref:
        ref.set_tuning("enc_census", 1)
        want = [ref.encode_block(sch.types, t) for t in blocks]
    with Context(0) as c:
        c.set_tuning("kernel_timing", 1)
        for j, t in enumerate(blocks):
            c.kernel_times()
            blk = c.encode_block(sch.types, t)
            kt = c.kernel_times()
            assert ("k_row_census" in kt) == (j == 0), f"block {j}: {sorted(kt)}"
            assert ("k_row_fixup" in kt) == (j > 0), f"block {j}: {sorted(kt)}"
            for f in FIELDS:
                assert getattr(blk, f) == getattr(want[j], f), f"block {j}: {f}"
    if rows == 4096:
        port = O.encode(sch, blocks[1])
        assert port.rc == 0
        assert G.split_header(port.data)[1] == want[1].data


def _wide_schema():
    return O.parse_desc(corpus.desc([("a", "text"), ("b", "int(11)"), ("c", "varchar(255)"), ("d", "text")]))


def _row(rng, length, tail=b""):
    """One 4-column row of `length` bytes (at least 12) whose last field ends in `tail`, right in front of the newline."""
    b = b"%d" % rng.randrange(1000)
    c = rng.choice([b"x", b"yy", b"zzz"])
    d = bytes(rng.choice(b"abcdef") for _ in range(rng.randrange(4))) + tail
    pad = max(1, length - len(b) - len(c) - len(d) - 4)
    a = bytes(rng.choice(b"ghijkl") for _ in range(pad))
    return b"\t".join([a, b, c, d]) + b"\n"


def _rows_to(rng, out: bytearray, end: int):
    """Rows until out has exactly `end` bytes (the last row absorbs the difference)."""
    while end - len(out) > 1400:
        out += _row(rng, rng.randrange(200, 1200))
    if end - len(out) >= 12:
        out += _row(rng, end - len(out))
    assert len(out) <= end


def _boundary_inputs():
    """Windows with row breaks, blank lines and backslash runs placed at 2 KiB tile boundaries."""
    rng = random.Random(7)
    T = 2048
    cases = []
    # a row longer than a tile (the tile in the middle owns no row), then a row starting exactly at t0
    t = bytearray(_row(rng, 300))
    t += _row(rng, 3 * T + 500)
    _rows_to(rng, t, 5 * T)
    _rows_to(rng, t, 7 * T)
    cases.append(("long_row_and_start_at_t0", bytes(t)))
    # a newline at t0 - 1 followed by blank lines across the boundary, and blank lines just in front of it
    t = bytearray()
    _rows_to(rng, t, T)
    t += b"\n\n\n"
    _rows_to(rng, t, 2 * T - 2)
    t += b"\n\n\n\n"
    _rows_to(rng, t, 4 * T)
    cases.append(("blank_lines_across_boundaries", bytes(t)))
    # odd and even backslash runs right in front of a newline at a boundary (odd: the newline is escaped)
    for k in range(1, 6):
        t = bytearray(_row(rng, 100))
        _rows_to(rng, t, T - 400)
        t += _row(rng, 400, tail=b"\\" * k)
        if k % 2:  # the newline is escaped: the last field goes on in the next line
            t += b"more\n"
        _rows_to(rng, t, 3 * T)
        cases.append((f"backslashes_{k}_before_boundary_newline", bytes(t)))
    # leading blank lines, longer than a tile
    t = bytearray(b"\n" * (T + 5))
    _rows_to(rng, t, 4 * T)
    cases.append(("leading_blank_lines", bytes(t)))
    # random rows, blank lines and backslash runs: every kind of byte lands on some boundary
    for s in range(6):
        r = random.Random(100 + s)
        t = bytearray()
        while len(t) < 40 * T:
            x = r.random()
            if x < 0.1:
                t += b"\n" * r.randrange(1, 4)
            elif x < 0.2:
                t += _row(r, r.randrange(20, 200), tail=b"\\" * r.randrange(0, 5, 2))
            else:
                t += _row(r, r.randrange(100, 5000))
        cases.append((f"random_{s}", bytes(t)))
    return cases


@pytest.mark.parametrize("tile", [2048, 4096])
def test_tile_boundaries(knobs, tile):
    ctx = knobs
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", tile)
    sch = _wide_schema()
    for name, tsv in _boundary_inputs():
        _same(ctx, sch.types, tsv, name)
        want = O.encode(sch, tsv)
        if want.rc == 0:
            got = _file(ctx, 0, sch, tsv)
            assert got == want.data, f"{name}: {G.first_diff(got, want.data)}"


@pytest.mark.parametrize("offset", [1, 3, 8, 13])
def test_misaligned_device_input(knobs, offset):
    import torch
    ctx = knobs
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", 2048)
    sch = _wide_schema()
    for name, tsv in _boundary_inputs()[-2:]:
        t = torch.zeros(len(tsv) + 128, dtype=torch.uint8, device="cuda")
        t[offset:offset + len(tsv)].copy_(torch.frombuffer(bytearray(tsv), dtype=torch.uint8))
        torch.cuda.synchronize()
        got = _same(ctx, sch.types, t.data_ptr() + offset, name, n=len(tsv), input_on_device=True)
        assert got[0]["data"] == ctx.encode_block(sch.types, tsv).data


def test_tail(knobs):
    """What follows the last row break: no final newline (more input follows or not), trailing newlines, no row at all."""
    ctx = knobs
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", 2048)
    sch = _wide_schema()
    rng = random.Random(3)
    body = bytearray()
    _rows_to(rng, body, 9000)
    body = bytes(body)
    unterminated = _row(rng, 3000)[:-1]
    for name, tsv in (("no_final_newline", body + unterminated), ("trailing_newlines", body + b"\n\n\n"),
                      ("short_tail", body + b"q"), ("tail_of_newline_and_bytes", body + b"\nab\tc"),
                      ("no_complete_row", unterminated), ("only_newlines", b"\n" * 5000),
                      ("blank_lines_then_partial_row", b"\n" * 3000 + unterminated)):
        for more in (False, True):
            r = _same(ctx, sch.types, tsv, f"{name} more_input_follows={more}", more_input_follows=more)
            if name in ("no_complete_row", "only_newlines", "blank_lines_then_partial_row"):
                assert r[0]["rows_in_buffer"] == 0 and r[0]["tsv_consumed"] == (0 if more else len(tsv))


def test_malformed_row_in_a_late_tile(knobs):
    ctx = knobs
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", 2048)
    sch = _wide_schema()
    rng = random.Random(5)
    t = bytearray()
    _rows_to(rng, t, 30000)
    t += b"only\ttwo\n"
    _rows_to(rng, t, 40000)
    t += b"a\tb\tc\td\te\n"
    _rows_to(rng, t, 50000)
    got = _same(ctx, sch.types, bytes(t), "malformed")
    assert got[1] is not None and got[1][0] == 3  # ZDWB_ERR_WRONG_COLUMNS
    want = O.encode(sch, bytes(t))
    assert want.rc == 15 and got[1][1] == want.bad_row


def test_blank_lines_beyond_the_row_limit_fall_back_to_the_census(knobs):
    """No row starts within 64 KiB in front of a tile (a long run of blank lines): the block is encoded with the census,
    still on the row-delta path, and the context's later blocks take the census too."""
    ctx = knobs
    sch = _wide_schema()
    rng = random.Random(13)
    wide = bytearray()
    _rows_to(rng, wide, 600000)
    gap = bytearray()
    _rows_to(rng, gap, 300000)
    gap += b"\n" * 70000
    _rows_to(rng, gap, len(gap) + 300000)
    ctx.set_tuning("enc_census", 1)
    want = ctx.encode_block(sch.types, bytes(gap))
    ctx.set_tuning("enc_census", -1)
    ctx.set_tuning("kernel_timing", 1)
    ctx.encode_block(sch.types, bytes(wide))
    for j, kernels in enumerate(({"k_row_fixup", "k_row_census"}, {"k_row_census"})):
        ctx.kernel_times()
        blk = ctx.encode_block(sch.types, bytes(gap))
        kt = ctx.kernel_times()
        assert kernels <= set(kt) and "k_tile_count" not in kt, f"block {j}: {sorted(kt)}"
        assert ("k_row_fixup" in kt) == (j == 0), f"block {j}: {sorted(kt)}"
        for f in FIELDS:
            assert getattr(blk, f) == getattr(want, f), f
    assert G.split_header(O.encode(sch, bytes(gap)).data)[1] == want.data


def test_slot_overflow_falls_back_to_the_census(knobs):
    """Short rows after a wide block: a tile holds more rows than its slots, the block is encoded with the census."""
    ctx = knobs
    ctx.set_tuning("kernel_timing", 1)
    sch = _wide_schema()
    rng = random.Random(9)
    wide = bytearray()
    _rows_to(rng, wide, 600000)
    mixed = bytearray()
    for part in range(2):  # rows of about 2 KB around 500 rows of 20 bytes (hundreds in one 8 KiB tile)
        while len(mixed) < 300000 * (part + 1) + 10000 * part:
            mixed += _row(rng, rng.randrange(1500, 2500))
        for _ in range(500 if part == 0 else 0):
            mixed += _row(rng, 20)
    ctx.set_tuning("enc_census", 1)
    want = [ctx.encode_block(sch.types, bytes(x)) for x in (wide, mixed)]
    ctx.set_tuning("enc_census", -1)
    ctx.encode_block(sch.types, bytes(wide))  # history from a wide delta block: the next block goes census-free
    ctx.kernel_times()
    blk = ctx.encode_block(sch.types, bytes(mixed))
    kt = ctx.kernel_times()
    assert "k_row_fixup" in kt and "k_row_census" in kt, sorted(kt)
    for f in FIELDS:
        assert getattr(blk, f) == getattr(want[1], f), f
    assert G.split_header(O.encode(sch, bytes(mixed)).data)[1] == blk.data


def test_hash_set_and_record_growth(knobs):
    """The retry loop of pass 1 (a hash set or record arrays that fill up) on the census-free path."""
    from zdw_b200 import Context
    ctx = knobs
    ctx.set_tuning("enc_delta", 1)
    # many distinct strings into a 2^10-slot hash set (a fresh context: no earlier block sizes it)
    sch = O.parse_desc(O.golden("analytics-hits.desc.sql"))
    tsv = O.golden("analytics-hits.sql")
    with Context(0) as c:
        c.set_tuning("enc_delta", 1)
        c.set_tuning("ht_initial_log2", 10)
        c.set_tuning("kernel_timing", 1)
        c.set_tuning("enc_census", 0)
        got = c.encode_block(sch.types, tsv)
        assert c.kernel_times()["k_pass1d"][0] >= 2
    c2 = _encode(ctx, 1, sch.types, tsv)[0]
    assert {f: getattr(got, f) for f in FIELDS} == c2
    # every field of every row changes: more records than a sixteenth of the bytes
    ncols = 250
    sch = O.parse_desc(corpus.desc([(f"c{i}", "int(11)") for i in range(ncols)]))
    tsv = b"".join(b"\t".join(b"%d" % ((r + i) % 10) for i in range(ncols)) + b"\n" for r in range(3000))
    with Context(0) as c:
        c.set_tuning("enc_delta", 1)
        c.set_tuning("kernel_timing", 1)
        c.set_tuning("enc_census", 0)
        got = c.encode_block(sch.types, tsv)
        assert c.kernel_times()["k_pass1d"][0] >= 2
    assert {f: getattr(got, f) for f in FIELDS} == _encode(ctx, 1, sch.types, tsv)[0]
    assert G.split_header(O.encode(sch, tsv).data)[1] == got.data


def test_trim(knobs):
    ctx = knobs
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", 2048)
    sch = _wide_schema()
    rng = random.Random(11)
    t = bytearray()
    while len(t) < 60000:
        r = _row(rng, rng.randrange(100, 3000))
        t += r.replace(b"\t", b"  \t", rng.randrange(3)) if rng.random() < 0.5 else r
    _same(ctx, sch.types, bytes(t), "trim", trim=True)
    want = O.encode(sch, bytes(t), trim=True)
    assert want.rc == 0
    assert _file(ctx, 0, sch, bytes(t), trim=True) == want.data
