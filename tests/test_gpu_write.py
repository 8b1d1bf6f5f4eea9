"""GPU tests of writing columns back to ZDW (zdwb_render_columns, write_table).  The references are the Python restatement
of the cell texts and rules (tests/render_util.py), the product's TSV decoder, and the C restatement of the encoder and
the decoder: a written file must be byte for byte the C restatement's encoding of the rendered text."""
import bz2
import ctypes as C
import gzip
import lzma
import os
import random
import subprocess

import pytest

import corpus
import gpuutil as G
import near_miss
import oracle as O
import recorded_runs as RR
import render_util as R
from columns_util import CHAR, DECIMAL, INT64_MIN, TEXT_LIKE, entries
from columns_util import render as decoder_text
from test_gpu_columns import MIXED, _mixed_tsv

pytestmark = pytest.mark.gpu

BAD_ARG = 4
BIN = O.ROOT / "zdw_b200" / "bin"


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


def host_dicts(types, dicts):
    """per column (dict bytes, entry offsets) on the host, None for non-text columns"""
    out, seen = [], {}
    for t, dd in zip(types, dicts):
        if dd is None or t not in TEXT_LIKE:
            out.append(None)
            continue
        key = (dd[0].data_ptr(), dd[1].data_ptr(), dd[0].numel(), dd[1].numel())
        if key not in seen:
            seen[key] = (bytes(dd[0].cpu().numpy().tobytes()), dd[1].cpu().tolist())
        out.append(seen[key])
    return out


def check_render(ctx, types, cells, dicts):
    """render_columns against the Python restatement: the same bytes, or ZDWB_ERR_BAD_ARG naming the same cell.
    Returns the rendered bytes (None when refused)."""
    from zdw_b200 import ZdwError
    cols = [c.cpu().tolist() for c in cells]
    hd = host_dicts(types, dicts)
    fault = R.check(types, cols, hd)
    if fault is None:
        ptr, n = ctx.render_columns(types, cells, dicts)
        got = G.dev_bytes(ptr, n) if n else b""
        want = R.render(types, cols, hd)
        assert got == want, G.first_diff(got, want)
        return got
    with pytest.raises(ZdwError) as ei:
        ctx.render_columns(types, cells, dicts)
    assert ei.value.code == BAD_ARG
    k, r, rule = fault
    assert f"column {k} row {r} " in ei.value.msg and R.RULE_WORDS[rule] in ei.value.msg, (fault, ei.value.msg)
    return None


def block_dicts(types, blk):
    return [(blk.dict, blk.entry_off) if types[c] in TEXT_LIKE else None for c in blk.columns]


def check_blocks(ctx, image, cols=None):
    """every block of the image through decode_columns and render_columns"""
    sch, _, hl = O.read_header(image)
    cols = list(range(sch.ncols)) if cols is None else cols
    types = [sch.types[c] for c in cols]
    pos, blocks = hl, []
    while True:
        blk = ctx.decode_columns(sch.types, image, cols, len(image) - pos, offset=pos)
        blocks.append((pos, blk, check_render(ctx, types, list(blk.values), block_dicts(sch.types, blk))))
        pos += blk.consumed
        if blk.is_last:
            return sch, blocks


def check_table(ctx, image):
    from zdw_b200 import read_table
    hdr, t = read_table(image)
    types = [hdr.types[c] for c in t.columns]
    return check_render(ctx, types, list(t.values), t.dicts)


CASES = [c for c in corpus.cases() if "expect_rc" not in c[3] and not c[0].startswith("d2_")]


def readable(r):
    """an image the decoders read (zero-byte rows at the end of a file are the reference's ROW_COUNT_ERR)"""
    return r.rc == 0 and r.total_rows > 0 and O.decode(r.data).rc == 0


def _case_image(case, rows_per_block=0):
    name, desc, tsv, opts = case
    return O.encode(O.parse_desc(desc), tsv, trim=bool(opts.get("trim")), rows_per_block=rows_per_block)


# ----------------------------------------------------------------------------- 1. against the Python restatement

@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_corpus_case_blocks_and_tables(ctx, case):
    r = _case_image(case)
    if not readable(r):
        return
    check_blocks(ctx, r.data)
    check_table(ctx, r.data)


@pytest.mark.parametrize("name", ["analytics-hits.zdw", "movie_tickets.zdw"])
def test_goldens(ctx, name):
    z = O.golden(name)
    check_blocks(ctx, z)
    check_table(ctx, z)


def mixed_image(n, seed, rows_per_block=0, metadata=None):
    sch = O.parse_desc(corpus.desc(MIXED))
    return sch, O.encode(sch, _mixed_tsv(n, seed), rows_per_block=rows_per_block, metadata=metadata)


@pytest.mark.parametrize("nrows", [0, 1, 31, 32, 33, 65])
def test_row_counts(ctx, nrows):
    import torch
    sch, r = mixed_image(max(nrows, 1), 3 + nrows)
    _, blocks = check_blocks(ctx, r.data)
    blk = blocks[0][1]
    types = sch.types
    cells = list(blk.values[:, :nrows])
    got = check_render(ctx, types, cells, block_dicts(types, blk))
    assert got is not None and got.count(b"\n") == nrows
    if nrows == 0:
        ptr, n = ctx.render_columns(types, [torch.empty(0, dtype=torch.int64, device="cuda")] * len(types),
                                    block_dicts(types, blk))
        assert n == 0


def test_one_column(ctx):
    import torch
    d, eo = R.make_dict([b"a", b"bb\\\\", b"c\\\td"])
    dd = (torch.tensor(list(d), dtype=torch.uint8, device="cuda"), torch.tensor(eo, dtype=torch.int64, device="cuda"))
    for t, vals, dicts in (([0], [0, 1, 2, 2, 0], [dd]), ([10], [0, 5, -1, 7], [None]), ([6], [ord("x"), 0x5C + 9 * 256], [None]),
                           ([15], [INT64_MIN, -1, 0], [None])):
        assert check_render(ctx, t, [torch.tensor(vals, dtype=torch.int64, device="cuda")], dicts) is not None
    assert check_render(ctx, [0], [torch.tensor([0, -1], dtype=torch.int64, device="cuda")], [dd]) is None


def test_near_miss_4096_columns(ctx):
    fam = near_miss.e2_families()[0]
    name, desc, tsv = fam[0], fam[1], fam[2]
    r = O.encode(O.parse_desc(desc), tsv)
    assert r.rc == 0
    sch, blocks = check_blocks(ctx, r.data)
    assert sch.ncols == 4096 and all(b[2] is not None for b in blocks)


def test_long_entries_at_every_alignment(ctx):
    """entries of 1 to 4000 bytes, starting at every offset mod 16 of the dictionary and of the row"""
    import torch
    rng = random.Random(7)
    lens = sorted({1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 63, 64, 65, 100, 255, 1000, 3999, 4000} | {rng.randint(1, 4000) for _ in range(20)})
    ents = sorted({bytes(rng.choice(b"abcXYZ \\\xff") for _ in range(L)).replace(b"\\", b"\\\\") for L in lens})
    ents = [e for e in ents if R.writable(e)]
    for pad in range(16):  # shifts every entry's alignment in the dictionary
        d, eo = R.make_dict([b"p" * (pad + 1)] + ents)
        dd = (torch.tensor(list(d), dtype=torch.uint8, device="cuda"), torch.tensor(eo, dtype=torch.int64, device="cuda"))
        n = 3 * len(ents)
        a = torch.tensor([rng.randrange(len(ents) + 1) for _ in range(n)], dtype=torch.int64, device="cuda")
        b = torch.tensor([rng.randrange(-1, len(ents) + 1) for _ in range(n)], dtype=torch.int64, device="cuda")
        lead = torch.tensor([rng.randrange(10 ** rng.randint(0, 6)) for _ in range(n)], dtype=torch.int64, device="cuda")
        for types, cells, dicts in (([0, 1], [a, b], [dd, dd]), ([7, 1, 0], [lead, b, a], [None, dd, dd]),
                                    ([1] * 6 + [9] * 6, [b] * 6 + [lead] * 6, [dd] * 6 + [None] * 6),
                                    ([1] * 20, [b] * 10 + [a] * 10, [dd] * 20)):
            assert check_render(ctx, types, cells, dicts) is not None


def test_shared_and_separate_dictionaries(ctx):
    import torch
    d1, e1 = R.make_dict([b"x", b"yy", b"zzz"])
    d2, e2 = R.make_dict([b"other", b"q\\\nr"])
    t = lambda v, dt=torch.int64: torch.tensor(v, dtype=dt, device="cuda")
    A = (t(list(d1), torch.uint8), t(e1))
    B = (t(list(d2), torch.uint8), t(e2))
    c = [t([0, 1, 2, -1]), t([2, 2, 0, 1]), t([1, 0, -1, 1]), t([0, 0, 1, 1])]
    assert check_render(ctx, [0, 1, 0, 18], c, [A, A, B, A]) is not None
    # one dictionary seen through two entry_off views of different length: not the same dictionary
    assert check_render(ctx, [0, 0], [t([2, 1, 0, 0]), t([1, 1, 0, 0])], [A, (A[0], A[1][:3])]) is not None


def c4_tsv(n_rows, block=0):
    import bench
    synth = bench.Synth()
    cap = synth.cap_for(n_rows)
    buf = (C.c_uint8 * cap)()
    n = synth.block_into(block, n_rows, C.addressof(buf), cap)
    return synth.schema.types, bytes((C.c_uint8 * n).from_address(C.addressof(buf)))


def test_c4_slice(ctx):
    types, tsv = c4_tsv(32768)
    z = ctx.encode_block(types, tsv).data
    cb = ctx.decode_columns(types, z, list(range(len(types))))
    got = check_render(ctx, types, list(cb.values), block_dicts(types, cb))
    assert got is not None
    # and back: the rendered text encodes to a block with the same cells
    blk = ctx.encode_block(types, got)
    cb2 = ctx.decode_columns(types, blk.data, list(range(len(types))))
    assert R.render(types, cb2.values.cpu().tolist(), host_dicts(types, block_dicts(types, cb2))) == got


# ----------------------------------------------------------------------------- 2. against the product's TSV decoder

def decoder_safe(types, blk):
    """no DECIMAL -1 and no INT64_MIN cell: the decoder's text is the rendered text"""
    v = blk.values
    for k, t in enumerate(types):
        if t == DECIMAL and bool((v[k] == -1).any()):
            return False
        if t in R.SIGNED and bool((v[k] == INT64_MIN).any()):
            return False
    return True


@pytest.mark.parametrize("source", ["corpus", "mixed", "goldens"])
def test_equals_the_tsv_decoder(ctx, source):
    cols = None
    if source == "corpus":
        images = [r.data for r in (_case_image(c) for c in CASES) if readable(r)]
    elif source == "mixed":
        images = [mixed_image(3000, 21, rows_per_block=500)[1].data]
        cols = [0, 1, 2, 3, 4, 5, 8, 9]  # (g is DECIMAL with empty cells, h holds INT64_MIN)
    else:
        images = [O.golden("analytics-hits.zdw"), O.golden("movie_tickets.zdw")]
    compared = 0
    for image in images:
        sch, blocks = check_blocks(ctx, image, cols)
        sel = list(range(sch.ncols)) if cols is None else cols
        ocol = [-1] * sch.ncols
        for k, c in enumerate(sel):
            ocol[c] = k
        for pos, blk, got in blocks:
            if got is None or not decoder_safe([sch.types[c] for c in sel], blk):
                continue
            want = ctx.decode_block(sch.types, image[pos:], out_col=ocol, n_out=len(sel)).tsv
            assert got == want, G.first_diff(got, want)
            compared += 1
    assert compared > 0


# ----------------------------------------------------------------------------- 3. files against the C restatement

def written(tmp_path, header, table, name="out.zdw", **kw):
    from zdw_b200 import write_table
    p = tmp_path / name
    write_table(p, header, table, **kw)
    return p.read_bytes()


def oracle_file(header, table, sizes):
    types = [header.types[c] for c in table.columns]
    sch = O.Schema([header.names[c] for c in table.columns], types, [header.charsize[c] for c in table.columns])
    tsv = R.render(types, table.values.cpu().tolist(), host_dicts(types, table.dicts))
    r = O.encode(sch, tsv, plan=[(s, 0) for s in sizes], metadata=header.metadata)
    assert r.rc == 0
    return r.data


@pytest.mark.parametrize("layout", ["1", "7", "1000", "source", "single"])
@pytest.mark.parametrize("meta", [False, True])
def test_files_against_the_oracle(ctx, tmp_path, layout, meta):
    from zdw_b200 import read_table
    sch, r = mixed_image(2500, 31, rows_per_block=300, metadata={"k": "v", "a": "zz"} if meta else None)
    hdr, t = read_table(r.data)
    assert bool(hdr.metadata) == meta and t.block_rows == [300] * 8 + [100]
    total = sum(t.block_rows)
    if layout == "source":
        kw, sizes = {}, t.block_rows
    elif layout == "single":
        kw, sizes = {"rows_per_block": total}, [total]
    else:
        rpb = int(layout)
        kw, sizes = {"rows_per_block": rpb}, [min(rpb, total - s) for s in range(0, total, rpb)]
    got = written(tmp_path, hdr, t, **kw)
    want = oracle_file(hdr, t, sizes)
    assert got == want, G.first_diff(got, want)
    if layout == "source" and meta:
        assert got == r.data  # the mixed rows are canonical: the file comes back unchanged


# ----------------------------------------------------------------------------- 4. round trips

def assert_same_table(a, b):
    import torch
    assert a.columns == b.columns or len(a.columns) == len(b.columns)
    assert torch.equal(a.values, b.values)
    assert a.block_rows == b.block_rows
    for x, y in zip(a.dicts, b.dicts):
        assert (x is None) == (y is None)
        if x is not None:
            assert torch.equal(x[0], y[0]) and torch.equal(x[1].to(torch.int64), y[1].to(torch.int64))


def random_table(rng, nrows, types):
    """a table built in torch: every text column its own dense, sorted dictionary, every cell writable"""
    import torch
    from zdw_b200 import ColumnTable
    vals, dicts = [], []
    pool = [b"a", b"b ", b"trailing  ", b"\\\t", b"x\\\ny", b"\\\\", b"\xff\xfe", b"0", b"-3", b"long" * 30]
    for t in types:
        if t in TEXT_LIKE:
            ents = sorted({b"".join(rng.choice(pool) for _ in range(rng.randint(1, 3))) for _ in range(rng.randint(1, 12))})
            ents = ents[:max(1, nrows)]
            codes = list(range(len(ents))) + [rng.randrange(-1, len(ents)) for _ in range(nrows - len(ents))]
            rng.shuffle(codes)
            d, eo = R.make_dict(ents)
            dicts.append((torch.tensor(list(d), dtype=torch.uint8, device="cuda"), torch.tensor(eo, dtype=torch.int64, device="cuda")))
            vals.append(codes[:nrows])
        elif t == CHAR:
            forms = [0, ord("q"), -1, -128, 127, 0x5C + 9 * 256, 0x5C + 10 * 256, 0x5C + 0x5C * 256, 0x5C - 256]
            vals.append([rng.choice(forms) for _ in range(nrows)])
            dicts.append(None)
        else:
            special = [0, 1, -1, INT64_MIN, (1 << 63) - 1]
            vals.append([rng.choice(special) if rng.random() < 0.5 else rng.randrange(-(1 << 40), 1 << 40) for _ in range(nrows)])
            dicts.append(None)
    v = torch.tensor(vals, dtype=torch.int64, device="cuda")
    return ColumnTable(v, dicts, list(range(len(types))), [nrows])


def test_round_trip_of_files(ctx, tmp_path):
    from zdw_b200 import read_table
    for image in (mixed_image(2500, 41, rows_per_block=300)[1].data, O.golden("movie_tickets.zdw")):
        hdr, t = read_table(image)
        _, back = read_table(written(tmp_path, hdr, t))
        assert_same_table(t, back)
        _, back = read_table(written(tmp_path, hdr, t, rows_per_block=1000))
        assert back.block_rows[0] == 1000
        back.block_rows = t.block_rows
        assert_same_table(t, back)


def test_round_trip_of_random_tables(tmp_path):
    from zdw_b200 import FileHeader, read_table
    rng = random.Random(43)
    all_types = sorted(R.KNOWN)
    for trial in range(12):
        types = all_types if trial % 3 == 0 else [rng.choice(all_types) for _ in range(rng.randint(2, 9))]
        nrows = rng.choice([1, 2, 50, 333])
        t = random_table(rng, nrows, types)
        hdr = FileHeader(11, {}, [f"c{k}" for k in range(len(types))], list(types), [0] * len(types), 0)
        sizes = [nrows] if nrows < 4 else [nrows // 3, nrows // 3, nrows - 2 * (nrows // 3)]
        t.block_rows = sizes
        _, back = read_table(written(tmp_path, hdr, t))
        assert_same_table(t, back)


def test_projections_and_reorderings(tmp_path):
    import torch
    from zdw_b200 import ColumnTable, read_table
    sch, r = mixed_image(700, 47, rows_per_block=100)
    hdr, t = read_table(r.data)
    for sel in ([3, 1], [9, 0, 5, 2], [0], [4, 8, 7]):
        sub = ColumnTable(t.values[sel], [t.dicts[k] for k in sel], [t.columns[k] for k in sel], t.block_rows)
        got = written(tmp_path, hdr, sub)
        h2, back = read_table(got)
        assert h2.names == [hdr.names[c] for c in sel] and h2.types == [hdr.types[c] for c in sel]
        assert torch.equal(back.values, sub.values)
        assert got == oracle_file(hdr, sub, t.block_rows)
        # against the C restatement's projected decode of the source
        ocol = [-1] * sch.ncols
        for k, c in enumerate(sel):
            ocol[c] = k
        src = O.decode(r.data, out_col=ocol, n_out=len(sel)).tsv
        if 6 not in sel:  # (DECIMAL -1 renders empty, the decoder prints 0.000000000000)
            assert O.decode(got).tsv == src


# ----------------------------------------------------------------------------- 5. identity on canonical input

def test_identity_on_canonical_corpus_files(tmp_path):
    from zdw_b200 import read_table
    same = 0
    for name, desc, tsv, opts in CASES:
        if opts.get("trim"):
            continue
        F = O.encode(O.parse_desc(desc), tsv)
        if not readable(F) or O.decode(F.data).tsv != tsv:
            continue
        hdr, t = read_table(F.data)
        hd = host_dicts([hdr.types[c] for c in t.columns], t.dicts)
        if R.check([hdr.types[c] for c in t.columns], t.values.cpu().tolist(), hd) is not None:
            continue
        assert written(tmp_path, hdr, t) == F.data, name
        same += 1
    assert same > 5


# ----------------------------------------------------------------------------- 6. readers

def test_written_files_decode_with_the_cli_and_the_reference(tmp_path):
    from zdw_b200 import read_table
    sch, r = mixed_image(1200, 53, rows_per_block=250)
    hdr, t = read_table(r.data)
    got = written(tmp_path, hdr, t, rows_per_block=333)
    hd = host_dicts(hdr.types, t.dicts)
    V = t.values.cpu().tolist()
    want_dec = b"".join(b"\t".join(decoder_text(ty, v, entries(*dd) if dd else []) for ty, v, dd in zip(hdr.types, row, hd))
                        + b"\n" for row in zip(*V))
    assert O.decode(got).tsv == want_dec
    if (BIN / "unconvertDWfile").exists():
        d = tmp_path / "cli"
        d.mkdir()
        (d / "x.zdw").write_bytes(got)
        p = subprocess.run([str(BIN / "unconvertDWfile"), "-q", "-", "x.zdw"], cwd=d, env=RR.env(), capture_output=True,
                           timeout=300)
        assert p.returncode == 0 and p.stdout == want_dec
    if O.have_ref():
        rc, out, _ = O.ref_decode(got)
        assert rc == 0 and out == want_dec


# ----------------------------------------------------------------------------- 7. errors

def test_errors_name_the_cell_and_the_context_recovers(ctx):
    import torch
    from zdw_b200 import ZdwError
    t = lambda v, dt=torch.int64: torch.tensor(v, dtype=dt, device="cuda")
    good_d, good_eo = R.make_dict([b"ok", b"a\tb", b"x\\", b"", b"fine"])
    dct, eo = t(list(good_d), torch.uint8), t(good_eo)
    dd = (dct, eo)
    nul_d = t(list(b"\0a\0b\0c\0"), torch.uint8)
    cases = [
        ([0, 7], [t([0, 0, 4, 1]), t([1, 2, 3, 4])], [dd, None], (0, 3, R.SEPARATOR)),
        ([0, 7], [t([0, 2, 0]), t([1, 2, 3])], [dd, None], (0, 1, R.BACKSLASH)),
        ([7, 0], [t([1, 2, 3]), t([0, 4, 3])], [None, dd], (1, 2, R.ENTRY)),
        ([0, 7], [t([0, 5, 0]), t([1, 2, 3])], [dd, None], (0, 1, R.CODE)),
        ([0, 7], [t([0, -2, 0]), t([1, 2, 3])], [dd, None], (0, 1, R.CODE)),
        ([7, 6], [t([1, 2, 3]), t([0, ord("a") + ord("b") * 256, 0])], [None, None], (1, 1, R.CHAR_FORM)),
        ([6, 6], [t([0, 0x5C, 9]), t([9, 0, 0])], [None, None], (0, 1, R.CHAR_FORM)),
        ([6], [t([ord("a"), 0])], [None], (0, 1, R.EMPTY_ROW)),
        ([1], [t([0, -1])], [dd], (0, 1, R.EMPTY_ROW)),
        ([1, 7], [t([1, 0]), t([1, 1])], [(nul_d, t([1, 5, 7]))], (0, 1, R.ENTRY)),
        ([1, 7], [t([0, 1]), t([1, 1])], [(dct, t([1, 4, 100]))], (0, 1, R.OFFSETS)),
        ([1, 7], [t([0, 1]), t([1, 1])], [(dct, t([1, 4, 2]))], (0, 1, R.OFFSETS)),
    ]
    for types, cells, dicts, fault in cases:
        dicts = list(dicts) + [None] * (len(types) - len(dicts))
        hd = host_dicts(types, dicts)
        assert R.check(types, [c.cpu().tolist() for c in cells], hd) == fault, fault
        check_render(ctx, types, cells, dicts)
        # the next call works
        assert check_render(ctx, [0, 7], [t([0, 4]), t([1, 2])], [dd, None]) == b"ok\t1\nfine\t2\n"
    # unreferenced bad entries are accepted
    assert check_render(ctx, [0], [t([0, 4, 0])], [dd]) == b"ok\nfine\nok\n"
    assert check_render(ctx, [0, 7], [t([0, 0]), t([1, 1])], [(dct, t([1, 4, 100])), None]) is not None
    # arguments
    for types, cells, dicts in (([], [], []), ([0, 7], [t([0]), t([1, 2])], [dd, None]), ([4, 7], [t([1]), t([1])], [None, None]),
                                ([5], [t([1])], [None]), ([7, 200], [t([1]), t([1])], [None, None])):
        with pytest.raises(ZdwError) as ei:
            ctx.render_columns(types, cells, dicts)
        assert ei.value.code == BAD_ARG
        assert check_render(ctx, [7], [t([5])], [None]) == b"5\n"
    # NULL pointers through the C ABI
    from zdw_b200 import capi
    L = capi.load_library()
    out = capi._RenderOut()
    tarr = (C.c_uint8 * 1)(7)
    sch = capi._Schema(1, C.cast(tarr, C.POINTER(C.c_uint8)))
    assert L.zdwb_render_columns(ctx._h, C.byref(sch), None, C.byref(out)) == BAD_ARG
    part = (capi._CodePart * 1)(capi._CodePart(None, None, 0, 0, None, 3))
    assert L.zdwb_render_columns(ctx._h, C.byref(sch), part, C.byref(out)) == BAD_ARG
    assert L.zdwb_render_columns(ctx._h, None, part, C.byref(out)) == BAD_ARG
    tarr2 = (C.c_uint8 * 1)(0)
    sch2 = capi._Schema(1, C.cast(tarr2, C.POINTER(C.c_uint8)))
    codes = t([0, 0, 0])
    part2 = (capi._CodePart * 1)(capi._CodePart(None, None, 2, 9, codes.data_ptr(), 3))
    assert L.zdwb_render_columns(ctx._h, C.byref(sch2), part2, C.byref(out)) == BAD_ARG
    assert check_render(ctx, [7], [t([5])], [None]) == b"5\n"


def test_write_table_rejections(tmp_path):
    import torch
    from zdw_b200 import ColumnTable, FileHeader, ZdwError, write_table
    hdr = FileHeader(11, {}, ["a", "b"], [7, 0], [0, 0], 0)
    d, eo = R.make_dict([b"x", b"y\tz"])
    dd = (torch.tensor(list(d), dtype=torch.uint8, device="cuda"), torch.tensor(eo, dtype=torch.int64, device="cuda"))
    v = torch.tensor([[1, 2, 3], [0, -1, 0]], dtype=torch.int64, device="cuda")
    p = tmp_path / "x.zdw"
    bad = [ColumnTable(v[:, :0], [None, dd], [0, 1], []),
           ColumnTable(v, [None, dd], [0, 1], [2]), ColumnTable(v, [None, dd], [0, 1], [0, 3]),
           ColumnTable(v.cpu(), [None, dd], [0, 1], [3]), ColumnTable(v.to(torch.int32), [None, dd], [0, 1], [3]),
           ColumnTable(v[0], [None], [0], [3]), ColumnTable(v, [None, dd], [0, 5], [3])]
    for tb in bad:
        with pytest.raises(ValueError):
            write_table(p, hdr, tb)
    with pytest.raises(ValueError):
        write_table(p, hdr, ColumnTable(v, [None, dd], [0, 1], [3]), rows_per_block=0)
    with pytest.raises(ValueError):
        write_table(tmp_path / "x.zdw.zst", hdr, ColumnTable(v, [None, dd], [0, 1], [3]))
    v2 = torch.tensor([[1, 2, 3], [0, 1, 0]], dtype=torch.int64, device="cuda")
    with pytest.raises(ZdwError) as ei:
        write_table(p, hdr, ColumnTable(v2, [None, dd], [0, 1], [3]))
    assert ei.value.code == BAD_ARG and "column 1 row 1 " in ei.value.msg


# ----------------------------------------------------------------------------- 8. buffer lifetime

def test_render_buffer_survives_other_calls(ctx):
    from zdw_b200 import read_table
    sch, r = mixed_image(400, 61)
    hdr, t = read_table(r.data)
    ptr, n = ctx.render_columns(hdr.types, t.values, t.dicts)
    want = G.dev_bytes(ptr, n)
    blk = ctx.encode_block(sch.types, _mixed_tsv(5000, 62))
    cb = ctx.decode_columns(sch.types, blk.data, list(range(sch.ncols)))
    ctx.merge_codes([(cb.dict, cb.entry_off, cb.values[1]), (cb.dict, cb.entry_off, cb.values[3])])
    ctx.decode_block(sch.types, blk.data)
    assert G.dev_bytes(ptr, n) == want
    enc = ctx.encode_block(hdr.types, ptr, n, input_on_device=True)
    assert enc.nrows == 400
    assert enc.data == r.data[O.read_header(r.data)[2]:]


# ----------------------------------------------------------------------------- 9. torch's stream

def test_write_table_waits_for_torchs_stream(tmp_path):
    """The cells are produced on torch's current stream behind a spin kernel: write_table must see the final values."""
    import torch
    from zdw_b200 import ColumnTable, read_table
    sch, r = mixed_image(3000, 71, rows_per_block=1000)
    hdr, t = read_table(r.data)
    want = written(tmp_path, hdr, t, name="want.zdw")
    zeros = torch.zeros_like(t.values)
    # allocated and the kernel loaded up front: an allocation or a module load could synchronise and drain the spin
    late = torch.empty_like(t.values)
    torch.add(zeros, t.values, out=late)
    late.zero_()
    torch.cuda.synchronize()
    torch.cuda._sleep(4_000_000_000)
    torch.add(zeros, t.values, out=late)  # queued behind the spin
    assert not torch.cuda.current_stream().query()
    got = written(tmp_path, hdr, ColumnTable(late, t.dicts, t.columns, t.block_rows))
    assert got == want


# ----------------------------------------------------------------------------- 10. compression

@pytest.mark.parametrize("suffix,opener", [(".gz", gzip.open), (".bz2", bz2.open), (".xz", lzma.open)])
def test_compressed_files(tmp_path, suffix, opener):
    from zdw_b200 import read_table, write_table
    sch, r = mixed_image(900, 81, rows_per_block=200)
    hdr, t = read_table(r.data)
    p = tmp_path / ("out.zdw" + suffix)
    write_table(p, hdr, t)
    with opener(p, "rb") as f:
        assert f.read() == r.data
    _, back = read_table(p)
    assert_same_table(t, back)
    assert os.path.getsize(p) < len(r.data)
