"""GPU tests of the columnar decode (zdwb_decode_columns): every cell, rendered the way the TSV decoder prints it, must
give the C restatement's (or the product's own) decoded text, and the dictionary must be the block's sorted entries."""
import gzip
import lzma
import random

import pytest

import corpus
import gpuutil as G
import oracle as O
from columns_util import DATETIME, DECIMAL, SHORT, entries, render

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


def entries_of(blk):
    """The block's dictionary entries, after checking its invariants."""
    if blk.dict.numel() == 0:
        return []
    d = bytes(blk.dict.cpu().numpy().tobytes())
    eo = blk.entry_off.cpu().tolist()
    assert eo[-1] == len(d)
    assert all(a < b for a, b in zip(eo, eo[1:])), "entry offsets not strictly increasing"
    ents = entries(d, eo)
    assert all(d[b - 1] == 0 for b in eo[1:]) and d[:1] == b"\0"
    assert all(a < b for a, b in zip(ents, ents[1:])), "dictionary entries not in strictly increasing byte order"
    return ents


def block_text(blk, types, cols):
    """Rows of the block as tab-separated text of the selected columns, rendered from the int64 cells."""
    assert tuple(blk.values.shape) == (len(cols), blk.nrows)
    ents = entries_of(blk)
    rendered = []
    for k, c in enumerate(cols):
        t = types[c]
        rendered.append([render(t, v, ents) for v in blk.values[k].cpu().tolist()])
    return b"".join(b"\t".join(row) + b"\n" for row in zip(*rendered)) if rendered and blk.nrows else b""


def oracle_text(image, cols, nc):
    ocol = [-1] * nc
    for k, c in enumerate(cols):
        ocol[c] = k
    want = O.decode(image, out_col=ocol, n_out=len(cols))
    return want


def decode_file_columns(ctx, image, cols):
    sch, _, hl = O.read_header(image)
    pos, blocks = hl, []
    while True:
        blk = ctx.decode_columns(sch.types, image, cols, len(image) - pos, offset=pos)
        blocks.append(blk)
        pos += blk.consumed
        if blk.is_last:
            break
    return sch, blocks, pos


def check_file(ctx, image, cols=None):
    from zdw_b200 import ZdwError
    sch, _, _ = O.read_header(image)
    cols = list(range(sch.ncols)) if cols is None else cols
    want = oracle_text(image, cols, sch.ncols)
    if want.rc == 8:  # zero-byte rows at the end of the file: ROW_COUNT_ERR in the reference
        with pytest.raises(ZdwError) as ei:
            decode_file_columns(ctx, image, cols)
        assert ei.value.code == 8
        return None
    assert want.rc == 0
    sch, blocks, pos = decode_file_columns(ctx, image, cols)
    assert pos == len(image)
    got = b"".join(block_text(b, sch.types, cols) for b in blocks)
    assert got == want.tsv, G.first_diff(got, want.tsv)
    return blocks


CASES = [c for c in corpus.cases() if "expect_rc" not in c[3]]
FAST = [c for c in CASES if not c[0].startswith("d2_")]
D2 = [c for c in CASES if c[0].startswith("d2_")]


def _image(case, rows_per_block=0):
    name, desc, tsv, opts = case
    return O.encode(O.parse_desc(desc), tsv, trim=bool(opts.get("trim")), rows_per_block=rows_per_block)


@pytest.mark.parametrize("case", FAST, ids=[c[0] for c in FAST])
def test_corpus_case_all_columns(ctx, case):
    r = _image(case)
    if r.rc != 0 or r.total_rows == 0:
        return
    check_file(ctx, r.data)


def test_corpus_tile_boundaries(ctx):
    for case in D2[::5]:
        r = _image(case)
        if r.rc == 0 and r.total_rows:
            check_file(ctx, r.data)


def test_golden_analytics_hits_all_columns(ctx):
    z = O.golden("analytics-hits.zdw")
    sch, _, _ = O.read_header(z)
    assert sch.ncols == 2086
    blocks = check_file(ctx, z)
    assert blocks[0].ncols_used == 256


def test_golden_movie_tickets(ctx):
    z = O.golden("movie_tickets.zdw")
    blocks = check_file(ctx, z)
    assert sum(b.nrows for b in blocks) == 524160
    sch, _, _ = O.read_header(z)
    assert {DECIMAL, DATETIME, SHORT} <= set(sch.types)


def test_random_subsets_in_random_order(ctx):
    rng = random.Random(5)
    z = O.golden("analytics-hits.zdw")
    sch, _, _ = O.read_header(z)
    for _ in range(4):
        cols = rng.sample(range(sch.ncols), 16)
        check_file(ctx, z, cols)
    img = _image(next(c for c in CASES if c[0] == "mixed_3000")).data
    s2, _, _ = O.read_header(img)
    for _ in range(4):
        cols = rng.sample(range(s2.ncols), rng.randint(1, s2.ncols))
        check_file(ctx, img, cols)


MIXED = [("a", "int(11)"), ("b", "varchar(32)"), ("c", "bigint(20) unsigned"), ("d", "text"), ("e", "char(1)"),
         ("f", "smallint(5) unsigned"), ("g", "decimal(24,12)"), ("h", "bigint(20)"), ("i", "datetime"),
         ("j", "varchar(8)")]


def _mixed_tsv(n, seed):
    rng = random.Random(seed)
    rows = []
    for r in range(n):
        rows.append(b"\t".join([
            str(rng.randint(-1000, 1000)).encode(),
            rng.choice([b"", b"alpha", b"beta", b"gamma%d" % rng.randint(0, 50)]),
            str(rng.choice([0, 1, 2 ** 64 - 1, rng.randint(0, 2 ** 63)])).encode(),
            rng.choice([b"", b"t" * rng.randint(1, 40)]),
            rng.choice([b"", b"x", b"\\\\", b"\\t", b"Q"]),
            str(rng.randint(0, 65535)).encode(),
            rng.choice([b"", b"1.500000000000", b"-2.250000000000"]),
            str(rng.choice([-(2 ** 63), 2 ** 63 - 1, -5, 0])).encode(),
            rng.choice([b"2024-01-01 00:00:00", b"1999-12-31 23:59:59"]),
            b"", ]))  # j: never used
    return b"\n".join(rows) + b"\n"


@pytest.mark.parametrize("nrows", [1, 31, 32, 33, 65])
def test_small_blocks_and_unused_columns(ctx, nrows):
    sch = O.parse_desc(corpus.desc(MIXED))
    r = O.encode(sch, _mixed_tsv(nrows, nrows))
    assert r.rc == 0
    blocks = check_file(ctx, r.data)
    assert blocks[0].ncols_used < sch.ncols  # j is not used in the block
    check_file(ctx, r.data, [9, 3, 0])


def test_value_carried_across_many_strips(ctx):
    """Column b is explicit in row 0 and row 300 only: rows 1-299 take it from strips far back."""
    sch = O.parse_desc(corpus.desc([("a", "int(11)"), ("b", "varchar(9)"), ("c", "bigint(20)")]))
    rows = [b"%d\t%s\t%d" % (i, b"first" if i < 300 else b"second", -7 if i < 150 else 9) for i in range(700)]
    r = O.encode(sch, b"\n".join(rows) + b"\n")
    blocks = check_file(ctx, r.data)
    assert blocks[0].strings(1) == [b"first"] * 300 + [b"second"] * 400
    check_file(ctx, r.data, [2, 1])


@pytest.mark.parametrize("rows_per_block", [1, 7, 1000])
def test_read_columns_multi_block_files(ctx, tmp_path, rows_per_block):
    from zdw_b200 import read_columns
    sch = O.parse_desc(corpus.desc(MIXED))
    r = O.encode(sch, _mixed_tsv(1500 if rows_per_block > 1 else 40, 7), rows_per_block=rows_per_block)
    assert r.rc == 0 and r.nblocks > 1
    names = ["d", "a", "e", "b", "h"]
    cols = [sch.names.index(n) for n in names]
    want = oracle_text(r.data, cols, sch.ncols)
    for suffix, data in (("", r.data), (".gz", gzip.compress(r.data)), (".xz", lzma.compress(r.data))):
        p = tmp_path / f"f.zdw{suffix}"
        p.write_bytes(data)
        hdr, blocks = read_columns(p, names)
        assert hdr.names == sch.names and len(blocks) == r.nblocks
        got = b"".join(block_text(b, sch.types, cols) for b in blocks)  # each block against its own dictionary
        assert got == want.tsv, G.first_diff(got, want.tsv)
    hdr, blocks = read_columns(r.data)
    assert len(blocks) == r.nblocks and blocks[0].values.shape[0] == sch.ncols


def test_c4_slice_against_the_products_tsv(ctx):
    import ctypes as C

    import bench
    synth = bench.Synth()
    types = synth.schema.types
    n_rows = 32768
    cap = synth.cap_for(n_rows)
    buf = (C.c_uint8 * cap)()
    n = synth.block_into(0, n_rows, C.addressof(buf), cap)
    tsv = bytes((C.c_uint8 * n).from_address(C.addressof(buf)))
    blk = ctx.encode_block(types, tsv)
    assert blk.nrows == n_rows
    z = blk.data
    probe = ctx.decode_columns(types, z, [0])
    nc = len(types)
    # the used columns, from the column sizes behind the dictionary: numRows u32 | longestLine u32 | isLast u8 | idxSize u8
    isz = z[9]
    dsize = int.from_bytes(z[10:10 + isz], "little") if isz else 0
    csize = z[10 + isz + dsize:10 + isz + dsize + nc]
    used = [c for c in range(nc) if csize[c]]
    assert len(used) == probe.ncols_used
    cb = ctx.decode_columns(types, z, used)
    ocol = [-1] * nc
    for k, c in enumerate(used):
        ocol[c] = k
    want = ctx.decode_block(types, z, out_col=ocol, n_out=len(used)).tsv
    got = block_text(cb, types, used)
    assert got == want, G.first_diff(got, want)
    # and the same for the whole row against the product's NUL-separated in-memory layout
    full = ctx.decode_block(types, z, separator=b"\0").tsv
    cb_all = ctx.decode_columns(types, z, list(range(nc)))
    ents = entries_of(cb_all)
    V = cb_all.values.cpu().tolist()
    rendered = [[render(types[c], v, ents) for v in V[c]] for c in range(nc)]
    assert b"".join(b"\0".join(row) + b"\0" for row in zip(*rendered)) == full


def test_device_resident_input(ctx):
    import torch
    z = O.golden("analytics-hits.zdw")
    sch, _, hl = O.read_header(z)
    cols = [5, 0, 2085, 17, 100]
    want = oracle_text(z, cols, sch.ncols).tsv
    for shift in (0, 1, 7):
        t = torch.zeros(len(z) + 64, dtype=torch.uint8, device="cuda")
        t[shift:shift + len(z)] = torch.frombuffer(bytearray(z), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        blk = ctx.decode_columns(sch.types, t.data_ptr() + shift + hl, cols, len(z) - hl, input_on_device=True)
        assert blk.consumed == len(z) - hl
        assert block_text(blk, sch.types, cols) == want


def test_errors(ctx):
    from zdw_b200 import ZdwError
    one = O.parse_desc(corpus.desc([("a", "varchar(9)")]))
    z = bytearray(O.encode(one, b"hello\nworld\n").data)
    s2, _, hl = O.read_header(bytes(z))
    assert z[-1] == 7  # the last row's 1-byte offset: "world" in "\0hello\0world\0"
    # past the dictionary
    bad = bytearray(z)
    bad[-1] = 0x7F
    with pytest.raises(ZdwError) as ei:
        ctx.decode_columns(s2.types, bytes(bad[hl:]), [0])
    assert ei.value.code == 6
    # into the middle of an entry: the TSV decoder prints the tail, a code cannot
    mid = bytearray(z)
    mid[-1] = 8
    assert O.decode(bytes(mid)).tsv == b"hello\norld\n"
    with pytest.raises(ZdwError) as ei:
        ctx.decode_columns(s2.types, bytes(mid[hl:]), [0])
    assert ei.value.code == 6
    assert ctx.decode_block(s2.types, bytes(mid[hl:])).tsv == b"hello\norld\n"
    # truncated blocks
    img = _image(next(c for c in CASES if c[0] == "mixed_3000")).data
    s3, _, hl3 = O.read_header(img)
    blk = img[hl3:]
    for cut in (5, 12, len(blk) // 2, len(blk) - 1):
        with pytest.raises(ZdwError) as ei:
            ctx.decode_columns(s3.types, blk[:cut], [0, 1])
        assert ei.value.code in (7, 8)
    # bad column lists
    for cols in ([], [s3.ncols], [1, 0, 1]):
        with pytest.raises(ZdwError) as ei:
            ctx.decode_columns(s3.types, blk, cols)
        assert ei.value.code == 4
    # the context still decodes rows afterwards
    assert ctx.decode_block(s3.types, blk).tsv == O.decode(img).tsv


def test_decode_block_after_decode_columns(ctx):
    z = O.golden("movie_tickets.zdw")
    sch, _, hl = O.read_header(z)
    ctx.decode_columns(sch.types, z, list(range(sch.ncols)), offset=hl)
    got, _, _ = G.decode_file_with_product(ctx, z)
    assert got == O.golden("movie_tickets.sql")


def test_zero_row_block(ctx):
    """A block of no rows: header, dictionary and column stats only."""
    sch = O.parse_desc(corpus.desc([("a", "varchar(9)"), ("b", "int(11)"), ("c", "varchar(9)")]))
    img = O.encode(sch, b"hello\t5\t\nworld\t7\t\n").data
    _, _, hl = O.read_header(img)
    z = bytearray(img[hl:])
    isz = z[9]
    dsize = int.from_bytes(z[10:10 + isz], "little")
    csize = z[10 + isz + dsize:10 + isz + dsize + sch.ncols]
    rows_base = 10 + isz + dsize + sch.ncols + 8 * sum(1 for x in csize if x)
    z[0:4] = (0).to_bytes(4, "little")  # numRows = 0, and no rows follow
    empty = bytes(img[:hl] + z[:rows_base])
    assert O.decode(empty).rc == 0 and O.decode(empty).tsv == b""
    blk = ctx.decode_columns(sch.types, empty, [2, 0, 1], offset=hl)
    assert (blk.nrows, blk.consumed, blk.is_last, blk.ncols_used) == (0, rows_base, True, 2)
    assert tuple(blk.values.shape) == (3, 0)
    assert entries_of(blk) == [b"hello", b"world"]
    assert ctx.decode_block(sch.types, empty[hl:]).consumed == rows_base


def test_copies_complete_with_work_queued_on_torchs_stream(ctx):
    """The tensors are copied out of the context before its next call re-uses the memory, even while torch's current
    stream is busy: a spin kernel holds that stream for about two seconds while the 215 blocks of a file are decoded.
    (The context is warmed up first: an allocation by the context or by torch's cache would synchronise the device and
    drain the spin before the blocks are decoded.)"""
    import torch
    sch = O.parse_desc(corpus.desc(MIXED))
    r = O.encode(sch, _mixed_tsv(1500, 11), rows_per_block=7)
    cols = [sch.names.index(n) for n in ("b", "a", "h")]
    want = oracle_text(r.data, cols, sch.ncols).tsv
    blocks = decode_file_columns(ctx, r.data, cols)[1]
    assert len(blocks) == r.nblocks == 215
    del blocks
    torch.cuda.synchronize()
    torch.cuda._sleep(4_000_000_000)
    blocks = decode_file_columns(ctx, r.data, cols)[1]
    assert not torch.cuda.current_stream().query(), "the spin ended before the blocks were decoded: nothing was tested"
    got = b"".join(block_text(b, sch.types, cols) for b in blocks)
    assert got == want, G.first_diff(got, want)


def test_device_input_needs_avail(ctx):
    with pytest.raises(ValueError):
        ctx.decode_columns([0], 12345, [0], input_on_device=True)
