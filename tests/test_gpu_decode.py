"""GPU parity tests of the decoder: product (CUDA, through the C ABI) vs oracle, bit-exact."""
import os
import random

import pytest

import corpus
import gpuutil as G
import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


CASES = [c for c in corpus.cases() if "expect_rc" not in c[3]]
FAST = [c for c in CASES if not c[0].startswith("d2_")]
D2 = [c for c in CASES if c[0].startswith("d2_")]


def _image(case):
    name, desc, tsv, opts = case
    sch = O.parse_desc(desc)
    r = O.encode(sch, tsv, trim=bool(opts.get("trim")))
    return r


def _check_case(ctx, case, **kw):
    from zdw_b200 import ZdwError
    r = _image(case)
    if r.rc != 0 or r.total_rows == 0:
        return
    want = O.decode(r.data)
    if want.rc == 8:  # zero-byte rows at end of file: ROW_COUNT_ERR in the reference
        with pytest.raises(ZdwError) as ei:
            G.decode_file_with_product(ctx, r.data, **kw)
        assert ei.value.code == 8
        return
    assert want.rc == 0
    got, nblocks, consumed = G.decode_file_with_product(ctx, r.data, **kw)
    assert got == want.tsv, f"{case[0]}: {G.first_diff(got, want.tsv)}"
    assert consumed == len(r.data)


@pytest.mark.parametrize("case", FAST, ids=[c[0] for c in FAST])
def test_corpus_case(ctx, case):
    _check_case(ctx, case)


def test_corpus_tile_boundaries(ctx):
    for case in D2[::5]:
        _check_case(ctx, case)


@pytest.mark.parametrize("name", ["test", "analytics-hits", "movie_tickets"])
def test_golden_configs(ctx, name):
    """The reference's own v9/v10 golden files decode to their source TSV."""
    z = O.golden(f"{name}.zdw")
    tsv = O.golden(f"{name}.sql")
    got, nblocks, consumed = G.decode_file_with_product(ctx, z)
    assert got == tsv, G.first_diff(got, tsv)
    assert consumed == len(z) and nblocks == 1


@pytest.mark.parametrize("tile", [256, 1024, 32768])
def test_row_boundary_tile_sizes(ctx, tile):
    """Small tiles force multi-level map composition; large tiles exercise the single-level path."""
    ctx.set_tuning("dec_tile_bytes", tile)
    try:
        for name in ("analytics-hits", "movie_tickets"):
            z = O.golden(f"{name}.zdw")
            got, _, _ = G.decode_file_with_product(ctx, z)
            want = O.golden(f"{name}.sql")
            assert got == want, G.first_diff(got, want)
        for case in FAST:
            if case[0].startswith(("mixed", "d5", "d8_used25")):
                _check_case(ctx, case)
    finally:
        ctx.set_tuning("dec_tile_bytes", 8192)


@pytest.mark.parametrize("rpb", [1, 7, 1000])
def test_multi_block(ctx, rpb):
    case = next(c for c in CASES if c[0] == "mixed_3000")
    sch = O.parse_desc(case[1])
    img = O.encode(sch, case[2], rows_per_block=rpb).data
    want = O.decode(img)
    got, nblocks, consumed = G.decode_file_with_product(ctx, img)
    assert got == want.tsv, G.first_diff(got, want.tsv)
    assert nblocks == want.nblocks and consumed == len(img)


def test_column_projection(ctx):
    """-c / -cx / -ce style output maps (UnconvertFromZDW.cpp:1113-1190) incl. blank padding columns."""
    rng = random.Random(3)
    for name in ("analytics-hits", "mixed_3000"):
        if name == "mixed_3000":
            case = next(c for c in CASES if c[0] == name)
            img = _image(case).data
        else:
            img = O.golden(f"{name}.zdw")
        sch, _, _ = O.read_header(img)
        nc = sch.ncols
        for trial in range(4):
            k = rng.randrange(1, min(nc, 12))
            cols = rng.sample(range(nc), k)
            n_out = k + (trial % 2)            # one blank (missing) column appended on odd trials
            out_col = [-1] * nc
            positions = list(range(n_out))
            rng.shuffle(positions)
            for c, p in zip(cols, positions):
                out_col[c] = p
            want = O.decode(img, out_col=out_col, n_out=n_out)
            got, _, _ = G.decode_file_with_product(ctx, img, out_col=out_col, n_out=n_out)
            assert got == want.tsv, f"{name} trial {trial}: {G.first_diff(got, want.tsv)}"


def test_in_memory_layout_and_row_offsets(ctx):
    """NUL separators + row offsets: what the row-at-a-time getRow API hands out."""
    case = next(c for c in CASES if c[0] == "mixed_3000")
    img = _image(case).data
    sch, _, hl = O.read_header(img)
    want = O.decode(img, sep=b"\0")
    blk = ctx.decode_block(sch.types, img[hl:], separator=b"\0", want_row_offsets=True)
    assert blk.tsv == want.tsv
    assert blk.row_off[0] == 0 and blk.row_off[-1] == len(want.tsv) and len(blk.row_off) == blk.nrows + 1
    rows = want.tsv.split(b"\0")
    # every row ends with a NUL and has ncols fields: offsets must land on row starts
    ncols = sch.ncols
    acc = 0
    for r in range(0, blk.nrows, 97):
        start = blk.row_off[r]
        fields = want.tsv[start:blk.row_off[r + 1]].split(b"\0")
        assert len(fields) == ncols + 1 and fields[-1] == b""


def test_device_resident_io(ctx):
    import torch
    z = O.golden("analytics-hits.zdw")
    sch, _, hl = O.read_header(z)
    for shift in (0, 1, 7):
        t = torch.zeros(len(z) + 64, dtype=torch.uint8, device="cuda")
        t[shift:shift + len(z)] = torch.frombuffer(bytearray(z), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        blk = ctx.decode_block(sch.types, t.data_ptr() + shift + hl, len(z) - hl, input_on_device=True, output_on_device=True)
        got = G.dev_bytes(blk.dev_ptr, blk.length)
        assert got == O.golden("analytics-hits.sql")
        assert blk.consumed == len(z) - hl


def test_truncated_and_corrupt(ctx):
    from zdw_b200 import ZdwError
    case = next(c for c in CASES if c[0] == "mixed_3000")
    img = _image(case).data
    sch, _, hl = O.read_header(img)
    blk = img[hl:]
    for cut in (5, 12, len(blk) // 2, len(blk) - 1):
        with pytest.raises(ZdwError) as ei:
            ctx.decode_block(sch.types, blk[:cut])
        assert ei.value.code in (7, 8)
    # corrupt: point a text value past the dictionary -> CORRUPTED_DATA_ERROR
    z = bytearray(O.encode(O.parse_desc(corpus.desc([("a", "varchar(9)")])), b"hello\nworld\n").data)
    s2, _, hl2 = O.read_header(bytes(z))
    z[-1] = 0x7F  # last row's 1-byte dictionary offset
    with pytest.raises(ZdwError) as ei:
        ctx.decode_block(s2.types, bytes(z[hl2:]))
    assert ei.value.code == 6
    assert O.decode(bytes(z)).rc == 9


def test_roundtrip_property_large_random(ctx):
    """Size-independent property: decode(encode(x)) == canonical(x) on a larger random table."""
    rng = random.Random(99)
    cols = [("a", "int(11)"), ("b", "varchar(32)"), ("c", "bigint(20) unsigned"), ("d", "text"), ("e", "char(1)"),
            ("f", "smallint(5) unsigned"), ("g", "decimal(24,12)")]
    words = [b"w%d" % i for i in range(2000)]
    rows = []
    for i in range(60000):
        rows.append(b"\t".join([b"%d" % rng.randrange(-10**6, 10**6), rng.choice(words), b"%d" % rng.randrange(1, 2**63),
                                rng.choice(words) + b" " + rng.choice(words), rng.choice([b"x", b"y", b"z"]),
                                b"%d" % rng.randrange(1, 65535), b"%d.%02d" % (rng.randrange(1000), rng.randrange(100))]))
    tsv = b"\n".join(rows) + b"\n"
    sch = O.parse_desc(corpus.desc(cols))
    img = G.encode_file_with_product(ctx, sch, tsv)
    got, _, _ = G.decode_file_with_product(ctx, img)
    assert got == tsv  # canonical numerics: lossless
    assert img == O.encode(sch, tsv).data


@pytest.mark.parametrize("delta,lanes,strip", [(0, 0, 0), (0, 8, 0), (0, 16, 0), (1, 32, 0), (1, 32, 3), (1, 0, 1)])
def test_row_writer_variants_forced(ctx, delta, lanes, strip):
    """The row writer has variants: for wide schemas rows assembled from the row before (dec_delta: unchanged stretches
    copied 16 bytes at a time, only changed items rendered), 8, 16 or 32 lanes per row, the strip length.  Every
    combination must write the oracle's rows: the whole corpus, the goldens, projections, the in-memory layout; short
    strips make the delta writer start over often.  The knobs of removed variants are unknown names."""
    from zdw_b200 import ZdwError
    for removed in ("dec_emit_words", "dec_readback_kernel"):
        with pytest.raises(ZdwError) as ei:
            ctx.set_tuning(removed, 1)
        assert ei.value.code == 4  # ZDWB_ERR_BAD_ARG
    ctx.set_tuning("dec_delta", delta)
    ctx.set_tuning("dec_group_lanes", lanes)
    ctx.set_tuning("dec_strip_rows", strip)
    try:
        for case in FAST:
            _check_case(ctx, case)
        for name in ("analytics-hits", "movie_tickets"):
            img = O.golden(f"{name}.zdw")
            want = O.decode(img)
            got, _, _ = G.decode_file_with_product(ctx, img)
            assert got == want.tsv, f"{name}: {G.first_diff(got, want.tsv)}"
        test_column_projection(ctx)
        test_in_memory_layout_and_row_offsets(ctx)
    finally:
        ctx.set_tuning("dec_delta", 1)
        ctx.set_tuning("dec_group_lanes", 0)
        ctx.set_tuning("dec_strip_rows", 0)


@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_row_group_width_forced(ctx, lanes):
    """The row kernels give a strip to 8, 16 or 32 lanes (narrow schemas: several rows per warp).  Every width must
    decode every schema: forced here on the whole corpus, the wide golden, projections and the in-memory layout."""
    ctx.set_tuning("dec_group_lanes", lanes)
    try:
        for case in FAST:
            _check_case(ctx, case)
        for name in ("analytics-hits", "movie_tickets"):
            img = O.golden(f"{name}.zdw")
            want = O.decode(img)
            got, _, _ = G.decode_file_with_product(ctx, img)
            assert got == want.tsv, f"{name}: {G.first_diff(got, want.tsv)}"
        test_column_projection(ctx)
        test_in_memory_layout_and_row_offsets(ctx)
    finally:
        ctx.set_tuning("dec_group_lanes", 0)
