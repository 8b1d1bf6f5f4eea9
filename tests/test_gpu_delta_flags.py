"""The repeat flags of the row-delta encoder, decided from each record's own row and the row before.

Pass 2 of the row-delta path sets column c's flag in row r from rows r and r-1 alone: no flag when the field's bytes
are equal; a text-like column whose bytes differ is always flagged; a number or CHAR cell is flagged when its pass-2
value v2 (0 for an empty field) differs from the row before's.  The host tests restate that rule in Python and check
it against the flags and values in the C restatement's (oracle.encode) row stream over the corpus, the near-miss
families and the inputs below, and show over every two-byte CHAR prefix that a non-zero v2 never equals the column's
base (colmin - 1), the one case in which the rule would need the column statistics.  The GPU tests compare the
encoder's bytes with the C restatement on the census and census-free paths, with 2 KiB tiles so that the cases sit
on tile borders and block starts."""
import random

import pytest

import corpus
import gpuutil as G
import near_miss as N
import oracle as O

CHAR = 6
M64 = (1 << 64) - 1


# ------------------------------------------------------------------------------------------------ the rule in Python

def _s8(b):
    return b - 256 if b >= 128 else b


def _char_v(f):
    """(v1, v2) of a CHAR cell: sign-extended first byte, plus the second byte * 256 always (v2) or only behind a
    backslash (v1, the value the column's minimum is taken over)"""
    b0 = _s8(f[0])
    b1 = _s8(f[1]) * 256 if len(f) > 1 else 0
    return (b0 + (b1 if f[0] == 0x5C else 0)) & M64, (b0 + b1) & M64


def _num(f):
    """strtoull over the field: white space, a sign, digits; overflow saturates, '-' negates modulo 2^64"""
    i = 0
    while i < len(f) and (f[i] == 32 or 9 <= f[i] <= 13):
        i += 1
    neg = i < len(f) and f[i] == 0x2D
    if i < len(f) and f[i] in b"+-":
        i += 1
    v = 0
    while i < len(f) and 0x30 <= f[i] <= 0x39:
        v = v * 10 + f[i] - 0x30
        i += 1
    if v > M64:
        return M64
    return (-v) & M64 if neg else v


def _v2(t, f):
    if not f:
        return 0
    return _char_v(f)[1] if t == CHAR else _num(f)


def rule_flag(t, old, new):
    """the flag of a used column from its field in the row before and in this row (b"" = empty)"""
    if old == new:
        return False
    if t in O.TEXT_LIKE:
        return True
    return _v2(t, old) != _v2(t, new)


def _split(buf, sep):
    """split at `sep` bytes behind an even number of backslashes"""
    out, s, bs = [], 0, 0
    for i, b in enumerate(buf):
        if b == sep and bs % 2 == 0:
            out.append(buf[s:i])
            s = i + 1
        bs = bs + 1 if b == 0x5C else 0
    return out, buf[s:]


def tsv_rows(tsv, ncols, trim):
    lines, _ = _split(tsv, 0x0A)  # (an unterminated last line is no row)
    rows = []
    for ln in lines:
        if not ln:
            continue  # a blank line
        head, last = _split(ln, 0x09)
        f = head + [last]
        assert len(f) == ncols
        rows.append([x.rstrip(b" ") if trim else x for x in f])
    return rows


def zdw_blocks(img):
    """(schema, [(used columns, column sizes, bases, dictionary, rows)]) of a file; a row is {used column index:
    value} of its flagged columns"""
    sch, _, p = O.read_header(img)
    nc = sch.ncols
    blocks = []
    while p < len(img):
        nrows = int.from_bytes(img[p:p + 4], "little")
        last = img[p + 8]
        idx = img[p + 9]
        if idx:
            total = int.from_bytes(img[p + 10:p + 10 + idx], "little")
            dic = img[p + 10 + idx:p + 10 + idx + total]
            q = p + 10 + idx + total
        else:
            dic, q = b"", p + 10
        sizes = list(img[q:q + nc])
        q += nc
        used = [c for c in range(nc) if sizes[c]]
        bases = [int.from_bytes(img[q + 8 * k:q + 8 * k + 8], "little") for k in range(len(used))]
        q += 8 * len(used)
        nflag = (len(used) + 7) // 8
        rows = []
        for _ in range(nrows):
            fl = img[q:q + nflag]
            q += nflag
            row = {}
            for u in range(len(used)):
                if fl[u >> 3] >> (u & 7) & 1:
                    sz = sizes[used[u]]
                    row[u] = int.from_bytes(img[q:q + sz], "little")
                    q += sz
            rows.append(row)
        blocks.append((used, sizes, bases, dic, rows))
        p = q
        if last:
            break
    assert p == len(img)
    return sch, blocks


def check_rule(desc, tsv, trim=False, rows_per_block=0, plan=None):
    """the rule restated gives every flag of the C restatement's row stream, and the flagged values are the fields'"""
    sch = O.parse_desc(desc)
    r = O.encode(sch, tsv, trim=trim, rows_per_block=rows_per_block, plan=plan)
    if r.rc != 0:
        return 0
    _, blocks = zdw_blocks(r.data)
    rows = tsv_rows(tsv, sch.ncols, trim)
    k, checked = 0, 0
    for used, sizes, bases, dic, brows in blocks:
        prev = [b""] * sch.ncols  # a block starts from empty columns
        for flags in brows:
            cur = rows[k]
            k += 1
            for u, c in enumerate(used):
                t = sch.types[c]
                want = rule_flag(t, prev[c], cur[c])
                assert (u in flags) == want, (k - 1, c, prev[c], cur[c])
                checked += 1
                if not want:
                    continue
                v = flags[u]
                if not cur[c]:
                    assert v == 0
                elif t in O.TEXT_LIKE:
                    assert v and dic[v:dic.index(b"\0", v)] == cur[c]
                else:
                    v2 = _v2(t, cur[c])
                    assert v == ((v2 - bases[u]) & M64 if v2 else 0) & ((1 << (8 * sizes[c])) - 1)
            prev = cur
    return checked


# ------------------------------------------------------------------------------------------------ inputs

INT_POOL = [b"", b"0", b"-0", b"00", b"07", b"7", b"+7", b" 7", b"x", b"-1", b"18446744073709551615",
            b"18446744073709551616", b"99"]
CHR3_POOL = [b"", b"ab", b"abc", b"abd", b"abe", b"a", b"b", b"\\a", b"\\ab", b"\\b", b"-", b"\xe9", b"\xe9x", b"\xe9xy",
             b"\xe9xz", b"0", b"00"]
# (char(1) is the CHAR type; wider char(n) columns are text-like.  Cells of one column may be longer than declared:
# "abc" / "abd" and "\\ab" / "\\ac" differ only behind the two bytes v2 is made of)
CHR1_POOL = [b"", b"a", b"ab", b"ac", b"abc", b"abd", b"b", b"\x01", b"\x80", b"\\a", b"\\ab", b"\\ac", b"\xe9x", b"\xe9xy",
             b"\xe9xz"]
ZERO_POOL = [b"", b"0", b"-0", b"00", b"+0", b"x"]  # all parse to 0: the column is unused in the block
TXT_POOL = [b"", b"x", b"y", b"x ", b"xy", b"  "]

FLAG_DESC = corpus.desc([("a", "int(11)"), ("b", "bigint(20) unsigned"), ("c", "char(3)"), ("d", "char(1)"),
                         ("z", "int(11)"), ("t", "varchar(20)"), ("e", "char(2)"), ("pad", "text"), ("k", "int(11)")])


def flag_rows(seed, n=400):
    """rows whose fields change often, mostly within the pools' near misses; the pad column makes rows 60 - 700
    bytes long, so that 2 KiB tiles hold zero to a few row starts"""
    rng = random.Random(seed)
    pools = [INT_POOL, INT_POOL, CHR3_POOL, CHR1_POOL, ZERO_POOL, TXT_POOL, CHR3_POOL]
    cur = [b""] * len(pools)
    pad = b"p"
    out = []
    for i in range(n):
        for c, pool in enumerate(pools):
            if rng.random() < 0.45:
                cur[c] = rng.choice(pool)
        if rng.random() < 0.3:
            pad = bytes(rng.choices(b"abcdefgh", k=rng.choice([1, 40, 300, 650])))
        out.append(b"\t".join(cur + [pad, b"%d" % (i // 7)]))
    return b"\n".join(out) + b"\n"


WIDE = 600
WIDE_DESC = corpus.desc([("w%d" % c, "int(11)" if c % 3 == 0 else ("char(2)" if c % 3 == 1 else "varchar(8)"))
                         for c in range(WIDE)])


def wide_rows(seed):
    """rows of 0, 31 - 33, 280 and 560 records: 280 fields in columns 0 - 279, then 280 other ones (280 fields become
    empty, 280 change), identical rows, and rows with 31, 32 or 33 fields changed (some only in their spelling)"""
    rng = random.Random(seed)

    def row(cols, tag):
        f = [b""] * WIDE
        for c in cols:
            f[c] = b"%d" % (c % 97 + tag) if c % 3 != 2 else b"s%d" % ((c + tag) % 50)
        return f

    a = list(range(280))
    b = list(range(280, 560))
    c = list(range(0, 560, 2))
    out = []
    for tag in range(1, 7):
        for cols in (a, a, b, b, c, a, b):
            f = row(cols, tag)
            out.append(f)
            for k in (31, 32, 33):
                g = list(f)
                for col in rng.sample(cols, k):
                    g[col] = (b"0" + g[col]) if col % 3 == 0 and rng.random() < 0.5 else b"%d" % (col % 89 + 200)
                out.append(g)
                out.append(list(g))
    return b"\n".join(b"\t".join(f) for f in out) + b"\n"


def _cases():
    yield "flags", FLAG_DESC, flag_rows(1), {}
    yield "flags_trim", FLAG_DESC, flag_rows(2), {"trim": True}
    yield "flags_cut", FLAG_DESC, flag_rows(3), {"rows_per_block": 37}
    yield "flags_plan", FLAG_DESC, flag_rows(4), {"plan": [(50, 3), (1, 5), (90, 0), (20, 8)]}
    yield "wide", WIDE_DESC, wide_rows(5), {}
    yield "wide_cut", WIDE_DESC, wide_rows(6), {"rows_per_block": 11}
    yield "wide_plan", WIDE_DESC, wide_rows(7), {"plan": [(20, 300), (9, 1), (40, 599)]}


CASES = {c[0]: c for c in _cases()}


# ------------------------------------------------------------------------------------------------ host checks

def test_char_v2_never_equals_the_base():
    """a non-zero v2 of a CHAR cell is never colmin - 1 of a column holding the cell: over every first and second
    byte (a missing second byte reads as NUL), against every value a column's minimum can take - the non-zero v1 of
    any cell, and no larger than the cell's own v1 when that is non-zero"""
    cells = [_char_v(bytes([b0, b1])) for b0 in range(256) for b1 in range(256)]
    mins = {v1 for v1, _ in cells if v1}
    for v1, v2 in cells:
        if v2 == 0:
            continue
        colmin = (v2 + 1) & M64
        assert not (colmin in mins and (v1 == 0 or colmin <= v1)), (v1, v2)


@pytest.mark.parametrize("name", list(CASES))
def test_rule_on_new_inputs(name):
    _, desc, tsv, opts = CASES[name]
    assert check_rule(desc, tsv, trim=bool(opts.get("trim")), rows_per_block=opts.get("rows_per_block", 0),
                      plan=opts.get("plan")) > 0


def test_rule_on_corpus_and_near_miss():
    n = 0
    for name, desc, tsv, opts in corpus.cases():
        if opts.get("rows_per_block") or opts.get("plan") or opts.get("heap_blocks") or opts.get("metadata"):
            continue
        n += check_rule(desc, tsv, trim=bool(opts.get("trim")))
    for name, desc, tsv, _, claims in N.encode_families():
        o = claims.get("opts", {})
        n += check_rule(desc, tsv, trim=bool(o.get("trim")), rows_per_block=o.get("rows_per_block", 0))
    assert n > 0


def test_bytes_changed_is_not_the_flag():
    """the inputs hold fields whose bytes change while the flag stays clear (else the GPU tests could not tell the
    rule from "bytes changed => flag")"""
    for name in ("flags", "wide"):
        _, desc, tsv, _ = CASES[name]
        sch = O.parse_desc(desc)
        rows = tsv_rows(tsv, sch.ncols, False)
        kinds = set()
        for p, r in zip(rows, rows[1:]):
            for c, t in enumerate(sch.types):
                if p[c] != r[c] and not rule_flag(t, p[c], r[c]):
                    kinds.add("char" if t == CHAR else "int")
        assert kinds == ({"char", "int"} if name == "flags" else {"int"}), (name, kinds)


# ------------------------------------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    try:
        yield c
    finally:
        c.close()


@pytest.fixture()
def knobs(ctx):
    ctx.set_tuning("enc_delta", 1)
    ctx.set_tuning("enc_dtile", 2048)
    ctx.set_tuning("kernel_timing", 1)
    yield ctx
    for k, v in (("enc_census", -1), ("enc_delta", -1), ("enc_dtile", 0), ("kernel_timing", 0)):
        ctx.set_tuning(k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("census", [1, 0], ids=["census", "census_free"])
@pytest.mark.parametrize("name", list(CASES))
def test_encode_matches_restatement(knobs, name, census):
    ctx = knobs
    _, desc, tsv, opts = CASES[name]
    sch = O.parse_desc(desc)
    trim, rpb, plan = bool(opts.get("trim")), opts.get("rows_per_block", 0), opts.get("plan")
    want = O.encode(sch, tsv, trim=trim, rows_per_block=rpb, plan=plan)
    assert want.rc == 0
    ctx.set_tuning("enc_census", census)
    ctx.kernel_times()
    got = G.encode_file_with_product(ctx, sch, tsv, trim=trim, rows_per_block=rpb, plan=plan)
    ran = set(ctx.kernel_times())
    assert got == want.data, f"{name}: {G.first_diff(got, want.data)}"
    assert {"k_pass1d", "k_p2d_rowlen", "k_p2d_emit"} <= ran and "k_pass1" not in ran, sorted(ran)
    if census == 0 and not rpb and not plan:
        assert "k_row_fixup" in ran and "k_row_census" not in ran, sorted(ran)
