"""Near-miss inputs (tests/near_miss.py) through the two paths that skip work on "same as the row before".

Encode: every E family against the C restatement byte for byte, with the row-delta pass 1 forced (8 and 32 KiB tiles)
and with the general one.  Kernel timing shows which pass 1 ran: a block the row-delta pass gives back would pass the
byte comparison without having tested it.  Decode: every D family with the delta row writer at strips of 1 .. 64 rows,
projections in file order (the only ones the delta writer takes), and the columnar decoder on the same images."""
from functools import lru_cache

import pytest

import gpuutil as G
import near_miss as N
import oracle as O

pytestmark = pytest.mark.gpu

ENC = {f[0]: f for f in N.encode_families()}
DEC = {f[0]: f for f in N.decode_families()}
STRIPS = [0, 1, 2, 3, 7, 32, 64]
ENC_MODES = {"delta_tile8k": (1, 8192), "delta_tile32k": (1, 32768), "general": (0, 0)}


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    c.set_tuning("kernel_timing", 1)
    try:
        yield c
    finally:
        c.set_tuning("kernel_timing", 0)
        c.close()


def _opts(fam):
    o = fam[4].get("opts", {})
    return bool(o.get("trim")), o.get("rows_per_block", 0)


@lru_cache(maxsize=None)
def _oracle_image(name):
    fam = ENC.get(name) or DEC[name]
    trim, rpb = _opts(fam)
    r = O.encode(O.parse_desc(fam[1]), fam[2], trim=trim, rows_per_block=rpb)
    assert r.rc == 0
    return r.data


def _ran(ctx):
    """names of the kernels launched since the last call"""
    return set(ctx.kernel_times())


@pytest.mark.parametrize("mode", list(ENC_MODES))
@pytest.mark.parametrize("name", list(ENC))
def test_encode_family(ctx, name, mode):
    _, desc, tsv, canonical, claims = ENC[name]
    delta, tile = ENC_MODES[mode]
    sch = O.parse_desc(desc)
    trim, rpb = _opts(ENC[name])
    want = _oracle_image(name)
    ctx.set_tuning("enc_delta", delta)
    ctx.set_tuning("enc_dtile", tile)
    try:
        _ran(ctx)
        got = G.encode_file_with_product(ctx, sch, tsv, trim=trim, rows_per_block=rpb)
        ran = _ran(ctx)
    finally:
        ctx.set_tuning("enc_delta", -1)
        ctx.set_tuning("enc_dtile", 0)
    assert got == want, f"{name} ({mode}): {G.first_diff(got, want)}"
    if delta:
        assert "k_pass1d" in ran and "k_pass1" not in ran, f"{name}: the row-delta pass 1 did not encode every block"
    else:
        assert "k_pass1" in ran and "k_pass1d" not in ran
    if canonical and mode == "delta_tile8k":
        back, _, _ = G.decode_file_with_product(ctx, got)
        assert back == N.expected_tsv(tsv), f"{name}: {G.first_diff(back, N.expected_tsv(tsv))}"


def _delta_decode(ctx, strip, fn):
    """fn() with the delta row writer forced (32 lanes a strip, `strip` rows a strip); checks that it wrote the rows"""
    ctx.set_tuning("dec_delta", 1)
    ctx.set_tuning("dec_group_lanes", 32)
    ctx.set_tuning("dec_strip_rows", strip)
    try:
        _ran(ctx)
        out = fn()
        ran = _ran(ctx)
    finally:
        ctx.set_tuning("dec_delta", 1)
        ctx.set_tuning("dec_group_lanes", 0)
        ctx.set_tuning("dec_strip_rows", 0)
    assert "k_dec_write_delta" in ran and "k_dec_write_rows" not in ran, sorted(ran)
    return out


@pytest.mark.parametrize("strip", STRIPS, ids=[f"strip{s}" for s in STRIPS])
@pytest.mark.parametrize("name", list(DEC))
def test_decode_family(ctx, name, strip):
    img = _oracle_image(name)
    want = O.decode(img)
    assert want.rc == 0 and want.tsv == N.expected_tsv(DEC[name][2])
    got, _, consumed = _delta_decode(ctx, strip, lambda: G.decode_file_with_product(ctx, img))
    assert got == want.tsv, f"{name} strip {strip}: {G.first_diff(got, want.tsv)}"
    assert consumed == len(img)


def _out_col(nc, cols):
    oc = [-1] * nc
    for k, c in enumerate(cols):
        oc[c] = k
    return oc


def _halves(name, nc):
    """about half the columns in file order (-c) and the complement (-cx); for D1 the halves its rows with 63, 64 and
    65 selected changes (and 40 more outside them) are built for"""
    even = sorted(N.D1_SEL) if name == "D1_change_counts" else list(range(0, nc, 2))
    return [("even", even), ("odd", [c for c in range(nc) if c not in set(even)])]


@pytest.mark.parametrize("strip", [0, 1, 7], ids=["strip0", "strip1", "strip7"])
@pytest.mark.parametrize("name", N.PROJECTED)
def test_projection_in_file_order(ctx, name, strip):
    img = _oracle_image(name)
    sch, _, hl = O.read_header(img)
    nc = sch.ncols
    for half, cols in _halves(name, nc):
        for blank in (0, 1):  # (one blank column appended: n_out = k + 1)
            oc, n_out = _out_col(nc, cols), len(cols) + blank
            want = O.decode(img, out_col=oc, n_out=n_out)
            assert want.rc == 0
            got, _, _ = _delta_decode(ctx, strip, lambda: G.decode_file_with_product(ctx, img, out_col=oc, n_out=n_out))
            assert got == want.tsv, f"{name} {half} blank={blank}: {G.first_diff(got, want.tsv)}"
        # the in-memory layout: NUL after every field, row offsets.  (The restatement's ordered output, like the
        # reference's, writes tabs whatever the separator; the families have no escaped tabs or newlines, so its rows
        # with every tab and newline made a NUL are the expected bytes.)
        oc, n_out = _out_col(nc, cols), len(cols) + 1
        want = O.decode(img, out_col=oc, n_out=n_out)
        nul = want.tsv.replace(b"\t", b"\0").replace(b"\n", b"\0")
        blk = _delta_decode(ctx, strip, lambda: ctx.decode_block(sch.types, img[hl:], separator=b"\0", want_row_offsets=True,
                                                                 out_col=oc, n_out=n_out))
        assert blk.tsv == nul, f"{name} {half} NUL: {G.first_diff(blk.tsv, nul)}"
        ends = [i + 1 for i, b in enumerate(want.tsv) if b == 10]
        assert blk.row_off == [0] + ends
        # a constant text at the blank position (the oracle's rows with the blank filled)
        fill = b"<fill %d>" % len(cols)
        exp = b"".join(r + fill + b"\n" for r in want.tsv.split(b"\n")[:-1])
        got, _, _ = _delta_decode(ctx, strip, lambda: G.decode_file_with_product(ctx, img, out_col=oc, n_out=n_out,
                                                                                 fills={len(cols): fill}))
        assert got == exp, f"{name} {half} fills: {G.first_diff(got, exp)}"


@pytest.mark.parametrize("name", list(DEC))
def test_columns(ctx, name):
    """The same images through zdwb_decode_columns: every column, and D1's half the projections select."""
    import test_gpu_columns as TC
    img = _oracle_image(name)
    TC.check_file(ctx, img)
    if name == "D1_change_counts":
        TC.check_file(ctx, img, cols=sorted(N.D1_SEL))
