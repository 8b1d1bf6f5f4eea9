"""GPU parity tests of the encoder: product (CUDA, through the C ABI) vs oracle, bit-exact."""
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


def _check_case(ctx, case, **tuning):
    name, desc, tsv, opts = case
    sch = O.parse_desc(desc)
    trim = bool(opts.get("trim"))
    want = O.encode(sch, tsv, trim=trim)
    from zdw_b200 import ZdwError
    if want.rc == 15:
        with pytest.raises(ZdwError) as ei:
            ctx.encode_block(sch.types, tsv, trim=trim)
        assert ei.value.code == 3, name
        assert ei.value.bad_row == want.bad_row, name
        return
    assert want.rc == 0
    got = G.encode_file_with_product(ctx, sch, tsv, trim=trim)
    assert got == want.data, f"{name}: {G.first_diff(got, want.data)}"


CASES = corpus.cases()
FAST = [c for c in CASES if not c[0].startswith("d2_")]
D2 = [c for c in CASES if c[0].startswith("d2_")]


@pytest.mark.parametrize("case", FAST, ids=[c[0] for c in FAST])
def test_corpus_case(ctx, case):
    _check_case(ctx, case)


def test_corpus_tile_boundaries(ctx):
    for case in D2:
        _check_case(ctx, case)


@pytest.mark.parametrize("name", ["test", "analytics-hits", "movie_tickets"])
def test_golden_configs(ctx, name):
    """BASELINE configs C1-C3: bit-exact against the reference's own golden .zdw files."""
    sch = O.parse_desc(O.golden(f"{name}.desc.sql"))
    tsv = O.golden(f"{name}.sql")
    want = O.golden_to_v11(O.golden(f"{name}.zdw"))
    got = G.encode_file_with_product(ctx, sch, tsv)
    assert got == want, G.first_diff(got, want)


@pytest.mark.parametrize("items", [4, 16])
@pytest.mark.parametrize("name", ["analytics-hits", "movie_tickets"])
def test_golden_radix_sort_path(ctx, name, items):
    """Force the large-dictionary (radix + refinement) sort - with either tile size of its passes (the library picks 16
    records per thread from two million records on) - and a tiny first hash set."""
    sch = O.parse_desc(O.golden(f"{name}.desc.sql"))
    tsv = O.golden(f"{name}.sql")
    want = O.golden_to_v11(O.golden(f"{name}.zdw"))
    ctx.set_tuning("small_sort_max", 0)
    ctx.set_tuning("sort_radix_items", items)
    ctx.set_tuning("ht_initial_log2", 10)
    try:
        got = G.encode_file_with_product(ctx, sch, tsv)
    finally:
        ctx.set_tuning("small_sort_max", 65536)
        ctx.set_tuning("sort_radix_items", 0)
        ctx.set_tuning("ht_initial_log2", 20)
    assert got == want, G.first_diff(got, want)


@pytest.mark.parametrize("items", [4, 16])
def test_corpus_radix_sort_path(ctx, items):
    ctx.set_tuning("small_sort_max", 0)
    ctx.set_tuning("sort_radix_items", items)
    ctx.set_tuning("ht_initial_log2", 10)
    try:
        for case in FAST:
            if case[0].startswith(("d7", "d9", "d14", "mixed", "d1_", "d8_used25")):
                _check_case(ctx, case)
    finally:
        ctx.set_tuning("small_sort_max", 65536)
        ctx.set_tuning("sort_radix_items", 0)
        ctx.set_tuning("ht_initial_log2", 20)


@pytest.mark.parametrize("rpb", [1, 7, 1000, 2999, 3000])
def test_multi_block_explicit_rows(ctx, rpb):
    case = next(c for c in CASES if c[0] == "mixed_3000")
    sch = O.parse_desc(case[1])
    want = O.encode(sch, case[2], rows_per_block=rpb)
    got = G.encode_file_with_product(ctx, sch, case[2], rows_per_block=rpb)
    assert got == want.data, G.first_diff(got, want.data)
    # and the oracle decodes the stitched multi-block file back to the source rows
    dec = O.decode(got)
    assert dec.rc == 0 and dec.tsv == O.decode(O.encode(sch, case[2]).data).tsv
    assert dec.nblocks == -(-3000 // rpb)


def test_device_resident_unaligned_input(ctx):
    """Input already in HBM at every alignment 0..16 of the first byte; output left in HBM."""
    import torch
    case = next(c for c in CASES if c[0] == "mixed_3000")
    sch = O.parse_desc(case[1])
    want = O.encode(sch, case[2]).data
    _, want_blk = G.split_header(want)
    tsv = case[2]
    for shift in (0, 1, 3, 8, 15, 16, 17):
        t = torch.zeros(len(tsv) + 64, dtype=torch.uint8, device="cuda")
        t[shift:shift + len(tsv)] = torch.frombuffer(bytearray(tsv), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        blk = ctx.encode_block(sch.types, t.data_ptr() + shift, len(tsv), input_on_device=True, output_on_device=True)
        got = G.dev_bytes(blk.dev_ptr, blk.length)
        assert got == want_blk, f"shift {shift}: {G.first_diff(got, want_blk)}"


def test_device_resident_unaligned_leading_empty_field(ctx):
    """An empty first field at offset 0 of a buffer that is not 16-byte aligned (offset 0 acts as a boundary)."""
    import torch
    sch = O.parse_desc(corpus.desc([("a", "varchar(8)"), ("b", "varchar(8)"), ("c", "int(11)")]))
    tsv = b"\tfoo\t1\n\tbar\t2\nx\t\t3\n"
    _, want_blk = G.split_header(O.encode(sch, tsv).data)
    for shift in (0, 1, 5, 15):
        t = torch.zeros(len(tsv) + 64, dtype=torch.uint8, device="cuda")
        t[shift:shift + len(tsv)] = torch.frombuffer(bytearray(tsv), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        blk = ctx.encode_block(sch.types, t.data_ptr() + shift, len(tsv), input_on_device=True, output_on_device=True)
        got = G.dev_bytes(blk.dev_ptr, blk.length)
        assert got == want_blk, f"shift {shift}: {G.first_diff(got, want_blk)}"


def test_empty_inputs(ctx):
    sch = O.parse_desc(corpus.desc([("a", "varchar(8)"), ("b", "int(11)")]))
    for tsv in (b"", b"\n\n\n", b"x"):
        blk = ctx.encode_block(sch.types, tsv)
        assert blk.nrows == 0 and blk.length == 0


@pytest.mark.parametrize("plan", [[(1000, 0)], [(1000, 3), (500, 1)], [(7, 8)], [(2999, 2)], [(1, 1), (1, 9), (1, 4)]])
def test_explicit_block_plan_with_spill(ctx, plan):
    """(rows, spilled columns) per block - the reference's interrupted row (SURVEY App. B-14) - against the oracle."""
    case = next(c for c in CASES if c[0] == "mixed_3000")
    sch = O.parse_desc(case[1])
    want = O.encode(sch, case[2], plan=plan).data
    got = G.encode_file_with_product(ctx, sch, case[2], plan=plan)
    assert got == want, G.first_diff(got, want)


def test_reproduces_a_file_the_reference_cut_on_its_own(ctx):
    """The compiled reference splits a dictionary-heavy input when it runs low on memory (--mem-limit); with the block
    plan recovered from that file (test_block_plan.memory_cut_file: the restatement's file for the reference's cut) the
    CUDA encoder writes the same bytes, spilled strings included."""
    import c5_check
    import test_block_plan as BP
    sch = O.parse_desc(c5_check.DESC)
    tsv, image = BP.memory_cut_file()
    plan = BP.recover_plan(sch, tsv, image)
    assert plan and any(spill for _, spill in plan)
    got = G.encode_file_with_product(ctx, sch, tsv, plan=plan)
    assert got == image, G.first_diff(got, image)


@pytest.mark.parametrize("variant,p2_rows", [(1, 0), (1, 3), (1, 1), (0, 0)])
def test_pass1_variants_forced(ctx, variant, p2_rows):
    """Pass 1 has a row-delta variant (wide rows: only fields that differ from the row before are parsed and recorded)
    and a general one; `enc_delta` forces either, `enc_p2_rows` the rows per pass-2 tile (small tiles: the carried-in
    column values cross many tile borders).  Both must write the reference's bytes for every corpus case, the goldens,
    multi-block cuts and block plans with spilled columns."""
    ctx.set_tuning("enc_delta", variant)
    ctx.set_tuning("enc_p2_rows", p2_rows)
    try:
        for case in CASES:
            _check_case(ctx, case)
        for name in ("test", "analytics-hits", "movie_tickets"):
            if name == "movie_tickets" and p2_rows == 1:
                continue  # 524 160 one-row tiles: covered by the other tile sizes
            sch = O.parse_desc(O.golden(f"{name}.desc.sql"))
            want = O.golden_to_v11(O.golden(f"{name}.zdw"))
            got = G.encode_file_with_product(ctx, sch, O.golden(f"{name}.sql"))
            assert got == want, f"{name}: {G.first_diff(got, want)}"
        case = next(c for c in CASES if c[0] == "mixed_3000")
        sch = O.parse_desc(case[1])
        for rpb in (1, 7, 1000):
            want = O.encode(sch, case[2], rows_per_block=rpb).data
            got = G.encode_file_with_product(ctx, sch, case[2], rows_per_block=rpb)
            assert got == want, f"rows_per_block {rpb}: {G.first_diff(got, want)}"
        for plan in ([(1000, 3), (500, 1)], [(7, 8)], [(1, 1), (1, 9), (1, 4)]):
            want = O.encode(sch, case[2], plan=plan).data
            got = G.encode_file_with_product(ctx, sch, case[2], plan=plan)
            assert got == want, f"plan {plan}: {G.first_diff(got, want)}"
    finally:
        ctx.set_tuning("enc_delta", -1)
        ctx.set_tuning("enc_p2_rows", 0)


@pytest.mark.parametrize("tile", [2048, 4096, 16384, 65536])
def test_row_delta_tile_sizes(ctx, tile):
    """The row-delta pass cuts small inputs into smaller tiles (8 KiB .. 32 KiB by input size, `enc_dtile` forces one):
    rows that start in one tile and end tiles later, reference rows far in front of a tile, tiles without a row start."""
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", tile)
    try:
        for case in CASES:
            if case[0].startswith(("d1_", "d2_", "d3_", "d4_", "d7", "d8_used25", "d11", "mixed", "trim")):
                _check_case(ctx, case)
        sch = O.parse_desc(O.golden("analytics-hits.desc.sql"))
        want = O.golden_to_v11(O.golden("analytics-hits.zdw"))
        got = G.encode_file_with_product(ctx, sch, O.golden("analytics-hits.sql"))
        assert got == want, G.first_diff(got, want)
        case = next(c for c in CASES if c[0] == "mixed_3000")
        sch = O.parse_desc(case[1])
        for plan in ([(1000, 3), (500, 1)], [(7, 8)]):
            want = O.encode(sch, case[2], plan=plan).data
            got = G.encode_file_with_product(ctx, sch, case[2], plan=plan)
            assert got == want, f"plan {plan}: {G.first_diff(got, want)}"
    finally:
        ctx.set_tuning("enc_delta", -1)
        ctx.set_tuning("enc_dtile", 0)


def test_row_delta_falls_back_when_a_row_does_not_fit(ctx):
    """A row with more non-empty fields than a warp's lists hold (and one longer than 64 KiB): the row-delta pass gives
    the block back and the general pass encodes it - same bytes either way."""
    ncols = 700
    sch = O.parse_desc(corpus.desc([(f"c{i}", "varchar(8)" if i % 3 else "int(11)") for i in range(ncols)]))
    rows = [b"\t".join(b"%d" % ((r * 7 + i) % 13 + 1) for i in range(ncols)) for r in range(40)]
    tsv = b"\n".join(rows) + b"\n"
    want = O.encode(sch, tsv).data
    ctx.set_tuning("enc_delta", 1)
    try:
        got = G.encode_file_with_product(ctx, sch, tsv)
        assert got == want, G.first_diff(got, want)
        sch2 = O.parse_desc(corpus.desc([("a", "text"), ("b", "int(11)")]))
        long_rows = b"x" * 70000 + b"\t5\n" + b"y\t6\n" * 10 + b"z" * 66000 + b"\t7\n"
        want2 = O.encode(sch2, long_rows).data
        ctx.set_tuning("enc_delta", 1)
        got2 = G.encode_file_with_product(ctx, sch2, long_rows)
        assert got2 == want2, G.first_diff(got2, want2)
    finally:
        ctx.set_tuning("enc_delta", -1)


@pytest.mark.parametrize("case", corpus.big_cases(), ids=[c[0] for c in corpus.big_cases()])
def test_dictionary_offset_width_edge_at_2_24(ctx, case):
    """App. D d9: 2^24 - 1 / 2^24 / 2^24 + 1 dictionary bytes (3- vs 4-byte offsets), encode and decode."""
    name, desc, tsv, _ = case
    sch = O.parse_desc(desc)
    want = O.encode(sch, tsv)
    got = G.encode_file_with_product(ctx, sch, tsv)
    assert got == want.data, f"{name}: {G.first_diff(got, want.data)}"
    back, nblocks, consumed = G.decode_file_with_product(ctx, got)
    assert back == tsv and nblocks == 1 and consumed == len(got)


def test_longest_line_is_cumulative_over_blocks(ctx):
    desc, tsv, rpb = corpus.later_block_long_line()
    sch = O.parse_desc(desc)
    want = O.encode(sch, tsv, rows_per_block=rpb).data
    for variant in (1, 0):
        ctx.set_tuning("enc_delta", variant)
        try:
            got = G.encode_file_with_product(ctx, sch, tsv, rows_per_block=rpb)
        finally:
            ctx.set_tuning("enc_delta", -1)
        assert got == want, G.first_diff(got, want)


@pytest.mark.parametrize("K", [2, 3])
def test_heap_blocks_cut_like_the_reference_model(ctx, K):
    """zdwb_encode_opts.heap_blocks = K: the block ends where the reference's string heap would open its K-th 64 MiB
    block (SURVEY 8f-1, App. B-14) - against the restatement's model of StringHeap, which test_block_plan.py pins to a file
    the compiled reference cut on its own.  Every block of the file is cut that way."""
    import c5_check
    sch = O.parse_desc(c5_check.DESC)
    tsv = c5_check.make_rows(1_300_000 if K == 2 else 1_700_000)
    want = O.encode(sch, tsv, heap_blocks=K)
    assert want.rc == 0 and want.nblocks >= 2
    out = bytearray(G.split_header(want.data)[0])
    pos, longest, blocks = 0, 0, 0
    while pos < len(tsv):
        blk = ctx.encode_block(sch.types, tsv[pos:], prev_longest_line=longest, heap_blocks=K)
        assert blk.nrows > 0
        out += blk.data
        longest = blk.longest_line
        pos += blk.tsv_consumed
        blocks += 1
        if blk.nrows == blk.rows_in_buffer:
            break
    assert blocks == want.nblocks
    assert bytes(out) == want.data, G.first_diff(bytes(out), want.data)


def test_heap_blocks_first_row_is_out_of_memory(ctx):
    import c5_check
    from zdw_b200 import ZdwError
    sch = O.parse_desc(c5_check.DESC)
    with pytest.raises(ZdwError) as ei:
        ctx.encode_block(sch.types, c5_check.make_rows(1000), heap_blocks=1)
    assert ei.value.code == 2  # ZDWB_ERR_OOM: the reference's OUT_OF_MEMORY (ConvertToZDW.cpp:824-834)
