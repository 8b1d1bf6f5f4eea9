"""GPU tests of the predicates over a dictionary (zdwb_match_like, zdwb_find_strings) and of zdw_b200.predicates (like,
isin, between).  The oracles are the Python restatement in tests/match_util.py (itself held to sqlite and bisect by
tests/test_match_host.py) and, for the table predicates, the C restatement's decoded text of every cell."""
import bisect
import ctypes as C
import random

import pytest

import corpus
import oracle as O
from columns_util import DATETIME, DECIMAL, TEXT_LIKE, entries, render
import match_util as M

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


def dev_dict(ents):
    """A dictionary of sorted entries on the device, laid out as a block's (empty tensors for no entries)."""
    import torch
    if not ents:
        return torch.empty(0, dtype=torch.uint8, device="cuda"), torch.empty(0, dtype=torch.int64, device="cuda")
    d, eo = M.dict_bytes(ents)
    return torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda(), torch.tensor(eo, dtype=torch.int64, device="cuda")


def esc(b: bytes, e: int = 0x5C) -> bytes:
    """b as a LIKE literal: its wildcards and escape bytes escaped."""
    return b"".join(bytes([e, c]) if c in (0x25, 0x5F, e) else bytes([c]) for c in b)


def check_like(ctx, ents, pattern, escape=b"\\", ignore_case=False, null_text=b""):
    import torch
    d, eo = dev_dict(ents)
    torch.cuda.synchronize()
    got = ctx.match_like(d, eo, pattern, escape=escape, ignore_case=ignore_case, null_text=null_text)
    assert got.dtype == torch.bool and got.numel() == len(ents) + 1
    e = None if escape is None else escape[0]
    want = [M.like(s, pattern, e, ignore_case) for s in ents + [null_text]]
    assert got.cpu().tolist() == want, (pattern, escape, ignore_case)
    return sum(want)


def _lengths_dict(rng):
    """Entries with bytes 0x01-0xFF ('%', '_', '\\' and high bytes included), lengths around 1, 15, 16, 17, 32 and up to
    several KiB."""
    ents = set()
    alpha = b"ab%_\\\x01\x7f\x80\xffAB"
    for L in (1, 2, 15, 16, 17, 31, 32, 33, 64, 255, 1000, 4096, 6000):
        for _ in range(4):
            ents.add(bytes(rng.choice(alpha) for _ in range(L)))
        ents.add(b"ab" * (L // 2) + b"a" * (L % 2))
    ents.update(bytes([b]) for b in range(1, 256))
    return sorted(ents)


def test_match_like_patterns(ctx):
    rng = random.Random(1)
    ents = _lengths_dict(rng)
    longest = max(len(e) for e in ents)
    pats = [b"", b"%", b"_", b"%%", b"__", b"%_%", b"a%", b"%a", b"%b%a%", b"a_b%", b"\\%", b"%\\%%", b"%\\_%", b"%\\\\%",
            b"_" * 16, b"_" * 17, b"%" + b"_" * 4096 + b"%", b"a" * (longest + 1), b"%" + b"x" * (longest + 1) + b"%",
            b"%\x80%", b"\xff", b"%\xff\xff%", b"%AB%", b"%ab%"]
    for e in rng.sample(ents, 40):  # patterns cut from the entries: matches
        a = rng.randint(0, len(e))
        b = rng.randint(a, min(len(e), a + 40))
        pats += [esc(e), esc(e[:a]) + b"%", b"%" + esc(e[a:b]) + b"%", b"%" + esc(e[b:]), b"_" * len(e),
                 esc(e[:a]) + b"%" + esc(e[b:])]
    matches = 0
    for p in pats:
        matches += check_like(ctx, ents, p)
        matches += check_like(ctx, ents, p, ignore_case=True)
    assert matches > 1000
    # no escape byte; a different escape byte
    for p in (b"a\\%", b"%\\%", b"\\", b"%\\"):
        check_like(ctx, ents, p, escape=None)
    for p in (b"%!%%", b"!_%", b"%!!%", b"a%!a"):
        check_like(ctx, ents, p, escape=b"!")
    check_like(ctx, ents + [b"\xff\xff!"], b"%!%", escape=b"!")


def test_match_like_sizes_and_null_text(ctx):
    for ents in ([], [b"x"], [b"X"]):
        for p in (b"", b"%", b"_", b"x", b"%X%"):
            for null in (b"", b"0.000000000000"):
                for ic in (False, True):
                    check_like(ctx, list(ents), p, ignore_case=ic, null_text=null)
    assert check_like(ctx, [], b"", null_text=b"") == 1
    assert check_like(ctx, [], b"0.0%", null_text=b"0.000000000000") == 1
    assert check_like(ctx, [b"0.5"], b"0.0%", null_text=b"") == 0


def test_match_like_random(ctx):
    rng = random.Random(7)
    for _ in range(40):
        ents = sorted({bytes(rng.choice(b"aAbB%_\\\xc3") for _ in range(rng.randint(1, 12))) for _ in range(rng.randint(1, 300))})
        for _ in range(10):
            p = b"".join(rng.choice([b"%", b"_", b"a", b"B", b"\\%", b"\\_", b"\\\\", b"\xc3"]) for _ in range(rng.randint(0, 6)))
            check_like(ctx, ents, p, ignore_case=rng.random() < 0.5)


def check_find(ctx, ents, queries):
    import torch
    d, eo = dev_dict(ents)
    torch.cuda.synchronize()
    rank, found = ctx.find_strings(d, eo, queries)
    assert rank.dtype == torch.int64 and found.dtype == torch.bool and rank.numel() == len(queries)
    want = [bisect.bisect_left(ents, q) for q in queries]
    assert rank.cpu().tolist() == want
    assert found.cpu().tolist() == [r < len(ents) and ents[r] == q for r, q in zip(want, queries)]


def test_find_strings_queries(ctx):
    rng = random.Random(2)
    ents = _lengths_dict(rng)
    qs = [b"", b"\0", b"\0\0", b"\xff", b"\xff" * 20, b"\x01", b"a" * 7000]
    for e in rng.sample(ents, 60):
        qs += [e, e[:-1], e + b"\0", e + b"\x01", e + b"\xff", e[:16], e[:17], e[:1] + b"\0"]
    qs += qs[:50]  # duplicates
    rng.shuffle(qs)
    check_find(ctx, ents, qs)
    for small in ([], [b"m"], [b"", b"a"]):
        check_find(ctx, small, [b"", b"m", b"a", b"z", b"\0", b"\xff"])
    check_find(ctx, ents, [])


def test_find_strings_c5_shaped(ctx):
    """About a million distinct 65-byte entries and a million queries, half of them present."""
    import torch
    rng = random.Random(5)
    n = 1 << 20
    ents = sorted({b"%065x" % rng.getrandbits(200) for _ in range(n)})
    d, eo = dev_dict(ents)
    qs = [ents[rng.randrange(len(ents))] if rng.random() < 0.5 else b"%065x" % rng.getrandbits(200) for _ in range(n)]
    torch.cuda.synchronize()
    rank, found = ctx.find_strings(d, eo, qs)
    want = [bisect.bisect_left(ents, q) for q in qs]
    assert rank.cpu().tolist() == want
    fw = [r < len(ents) and ents[r] == q for r, q in zip(want, qs)]
    assert found.cpu().tolist() == fw and sum(fw) > n // 3
    flags = ctx.match_like(d, eo, b"%abc%")
    assert flags[:-1].cpu().tolist() == [b"abc" in e for e in ents]


# ----------------------------------------------------------------------------- errors

def test_errors_and_recovery(ctx):
    import torch
    from zdw_b200 import ZdwError, capi
    good = [b"a", b"b", b"c"]
    d, eo = dev_dict(good)

    def fails(call, code, text):
        torch.cuda.synchronize()
        with pytest.raises(ZdwError) as ei:
            call()
        assert ei.value.code == code, ei.value
        assert text in ei.value.msg, ei.value.msg
        check_like(ctx, good, b"%b%")  # the context works normally at its next call
        check_find(ctx, good, [b"b", b"bb"])

    L = ctx._L
    part = capi._CodePart(d.data_ptr(), eo.data_ptr(), 3, d.numel(), None, 0)
    opts = capi._LikeOpts(b"%", 1, b"", 0, 0x5C, 0)
    q = capi._Strings(None, 0, None, 0)
    mo, fo = capi._MatchOut(), capi._FindOut()
    # NULL pointers
    assert L.zdwb_match_like(ctx._h, None, C.byref(opts), C.byref(mo)) == 4
    assert L.zdwb_match_like(ctx._h, C.byref(part), None, C.byref(mo)) == 4
    assert L.zdwb_find_strings(ctx._h, None, C.byref(q), C.byref(fo)) == 4
    assert L.zdwb_find_strings(ctx._h, C.byref(part), None, C.byref(fo)) == 4
    for bad in (capi._CodePart(None, eo.data_ptr(), 3, d.numel(), None, 0), capi._CodePart(d.data_ptr(), None, 3, d.numel(), None, 0)):
        assert L.zdwb_match_like(ctx._h, C.byref(bad), C.byref(opts), C.byref(mo)) == 4
        assert L.zdwb_find_strings(ctx._h, C.byref(bad), C.byref(q), C.byref(fo)) == 4
    assert L.zdwb_match_like(ctx._h, C.byref(part), C.byref(capi._LikeOpts(None, 3, b"", 0, 0x5C, 0)), C.byref(mo)) == 4
    assert L.zdwb_match_like(ctx._h, C.byref(part), C.byref(capi._LikeOpts(b"%", 1, None, 2, 0x5C, 0)), C.byref(mo)) == 4
    assert L.zdwb_match_like(ctx._h, C.byref(part), C.byref(capi._LikeOpts(b"%", 1, b"", 0, 256, 0)), C.byref(mo)) == 4
    assert L.zdwb_find_strings(ctx._h, C.byref(part), C.byref(capi._Strings(None, 0, None, 2)), C.byref(fo)) == 4
    assert L.zdwb_find_strings(ctx._h, C.byref(part), C.byref(capi._Strings(None, 5, eo.data_ptr(), 1)), C.byref(fo)) == 4
    check_like(ctx, good, b"%")
    # a pattern that ends in a lone escape byte
    fails(lambda: ctx.match_like(d, eo, b"ab\\"), 4, "lone escape")
    fails(lambda: ctx.match_like(d, eo, b"ab!", escape=b"!"), 4, "lone escape")
    # entry offsets: not increasing, past dict_bytes; the lowest entry at fault is named
    for offs, low in (([1, 3, 3, 7], 1), ([1, 3, 99, 7], 1), ([1, 5, 3, 7], 1), ([1, 3, 5, 8], 2), ([9, 3, 5, 7], 0)):
        bad = torch.tensor(offs, dtype=torch.int64, device="cuda")
        fails(lambda: ctx.match_like(d, bad, b"%"), 4, f"entry {low} has offsets")
        fails(lambda: ctx.find_strings(d, bad, [b"a"]), 4, f"entry {low} has offsets")
    # entries not strictly increasing: equal, descending, past the prefix key; the lowest is named
    for ents, low in (([b"a", b"a"], 1), ([b"b", b"a"], 1), ([b"a", b"c", b"b", b"a"], 2),
                      ([b"x" * 20 + b"b", b"x" * 20 + b"a"], 1), ([b"ab", b"a"], 1)):
        dd, ee = dev_dict(ents)
        fails(lambda: ctx.find_strings(dd, ee, []), 4, f"entry {low} is not greater")
        check_like(ctx, ents, b"a%")  # LIKE does not need the order
    # query offsets that decrease or run past the buffer
    qb = torch.tensor(list(b"abcdef"), dtype=torch.uint8, device="cuda")
    for offs, low in (([0, 2, 1, 3], 1), ([0, 2, 7], 1), ([3, 2, 4], 0), ([0, 6, 6, 9], 2)):
        qo = torch.tensor(offs, dtype=torch.int64, device="cuda")
        qq = capi._Strings(qb.data_ptr(), 6, qo.data_ptr(), len(offs) - 1)
        torch.cuda.synchronize()
        assert L.zdwb_find_strings(ctx._h, C.byref(part), C.byref(qq), C.byref(fo)) == 4
        assert f"query {low} has offsets" in ctx.last_error(), ctx.last_error()
        check_find(ctx, good, [b"c"])
    qo = torch.tensor([0, 2, 2, 6], dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    assert L.zdwb_find_strings(ctx._h, C.byref(part), C.byref(capi._Strings(qb.data_ptr(), 6, qo.data_ptr(), 3)), C.byref(fo)) == 0
    with pytest.raises(ValueError):
        ctx.match_like(d, eo, b"%", escape=b"ab")


# ----------------------------------------------------------------------------- the table predicates

def host_table(image, names=None):
    """read_table of the image, and the text of every cell of its text-like columns, rendered from the table and held to
    the C restatement's decoded text of the same columns."""
    from zdw_b200 import read_table
    sch, _, _ = O.read_header(image)
    names = [n for n, t in zip(sch.names, sch.types) if t in TEXT_LIKE] if names is None else names
    if not names:
        return None, None, {}
    hdr, t = read_table(image, names)
    ocol = [-1] * sch.ncols
    for k, c in enumerate(t.columns):
        ocol[c] = k
    want = O.decode(image, out_col=ocol, n_out=len(names))
    assert want.rc == 0
    V = t.values.cpu().tolist()
    texts = {}
    for k, c in enumerate(t.columns):
        ents = entries(bytes(t.dicts[k][0].cpu().numpy().tobytes()), t.dicts[k][1].cpu().tolist()) if t.dicts[k] else []
        texts[k] = [render(sch.types[c], v, ents) for v in V[k]]
    got = b"".join(b"\t".join(row) + b"\n" for row in zip(*texts.values())) if V and V[0] else b""
    assert got == want.tsv
    return hdr, t, texts


def _mask(texts, pred):
    """pred of every text, computed once per distinct text"""
    cache = {s: pred(s) for s in set(texts)}
    return [cache[s] for s in texts]


def check_predicates(hdr, t, texts, rng, n=1):
    """like, isin and between on every text column against the host's answer from each cell's text; n picks of the
    column's own strings make the patterns, sets and ranges."""
    import torch
    from zdw_b200 import between, isin, like
    for k, tx in texts.items():
        distinct = sorted(set(tx))
        picks = [rng.choice(distinct) for _ in range(n)]
        pats = [b"%", b"_%"] + [esc(s[:3]) + b"%" for s in picks] + [b"%" + esc(s[1:4]) + b"%" for s in picks]
        for i, p in enumerate(pats):
            ic = i % 2 == 1
            got = like(hdr, t, k, p, ignore_case=ic)
            assert got.dtype == torch.bool and got.device == t.values.device
            assert got.cpu().tolist() == _mask(tx, lambda s: M.like(s, p, 0x5C, ic)), (k, p, ic)
        null = b"0.000000000000" if hdr.types[t.columns[k]] == DECIMAL else b""
        for st in ([], [null] + picks, picks + [b"\xff", b"\0", null + b"x"] + [s + b"\0" for s in picks]):
            ss = set(st)
            assert isin(hdr, t, k, st).cpu().tolist() == [s in ss for s in tx], (k, st)
        for _ in range(n):
            lo, hi = sorted([rng.choice(distinct), rng.choice(distinct)])
            for a, b in ((lo, hi), (hi + b"\0", lo), (null, null)):
                assert between(hdr, t, k, a, b).cpu().tolist() == [a <= s <= b for s in tx], (k, a, b)


CASES = [c for c in corpus.cases() if "expect_rc" not in c[3]]


def test_corpus_cases():
    rng = random.Random(11)
    checked = 0
    for name, desc, tsv, opts in CASES:
        sch = O.parse_desc(desc)
        if not any(t in TEXT_LIKE for t in sch.types):
            continue
        r = O.encode(sch, tsv, trim=bool(opts.get("trim")))
        if r.rc != 0 or r.total_rows == 0 or O.decode(r.data).rc != 0:  # (a file the decoder refuses has no table)
            continue
        hdr, t, texts = host_table(r.data)
        check_predicates(hdr, t, texts, rng)
        checked += 1
    assert checked > 50


@pytest.mark.parametrize("name", ["analytics-hits", "movie_tickets"])
def test_goldens(name, tmp_path):
    image = O.golden(f"{name}.zdw")
    sch, _, _ = O.read_header(image)
    text = [n for n, ty in zip(sch.names, sch.types) if ty in TEXT_LIKE]
    rng = random.Random(3)
    if len(text) > 12:  # analytics-hits: ten text columns and its DATETIME and DECIMAL ones
        text = rng.sample(text, 10) + [n for n, y in zip(sch.names, sch.types) if y in (DATETIME, DECIMAL)]
    names = text
    hdr, t, texts = host_table(image, list(dict.fromkeys(names)))
    types = {hdr.types[c] for c in t.columns}
    if name == "analytics-hits":
        assert DATETIME in types and DECIMAL in types
    check_predicates(hdr, t, texts, rng, 3 if name == "analytics-hits" else 1)
    for k, c in enumerate(t.columns):
        if hdr.types[c] == DATETIME:
            tx = texts[k]
            lo, hi = b"2000-01-01", b"2100-01-01 23:59:59"
            from zdw_b200 import between
            assert between(hdr, t, k, lo, hi).cpu().tolist() == [lo <= s <= hi for s in tx]
    if name == "analytics-hits":
        # its DECIMAL column holds 1.000000000000 in every row: empty every seventh cell of it (code -1, which the file
        # stores as an empty field and the decoder prints as 0.000000000000) and check the predicates on that file
        from zdw_b200 import ColumnTable, write_table
        k = next(k for k, c in enumerate(t.columns) if hdr.types[c] == DECIMAL)
        values = t.values.clone()
        values[k, ::7] = -1
        path = tmp_path / "nulls.zdw"
        write_table(path, hdr, ColumnTable(values, t.dicts, t.columns, t.block_rows))
        hdr2, t2, texts2 = host_table(path.read_bytes())
        k2 = next(k for k, c in enumerate(t2.columns) if hdr2.types[c] == DECIMAL)
        assert -1 in t2.values[k2].tolist() and b"0.000000000000" in texts2[k2]
        check_predicates(hdr2, t2, {k2: texts2[k2]}, rng, 2)


def test_block_dictionary_through_the_context(ctx):
    from zdw_b200 import read_columns
    from test_gpu_columns import MIXED, _mixed_tsv
    sch = O.parse_desc(corpus.desc(MIXED))
    r = O.encode(sch, _mixed_tsv(900, 5), rows_per_block=300)
    names = [n for n, ty in zip(sch.names, sch.types) if ty in TEXT_LIKE]
    _, blocks = read_columns(r.data, names)
    assert len(blocks) == 3
    for b in blocks:
        ents = entries(bytes(b.dict.cpu().numpy().tobytes()), b.entry_off.cpu().tolist())
        for k, n in enumerate(names):
            typ = sch.types[sch.names.index(n)]
            null = b"0.000000000000" if typ == DECIMAL else b""
            tx = [render(typ, v, ents) for v in b.values[k].cpu().tolist()]
            for p in (b"%a%", b"t%", b"%.5%", b""):
                flags = ctx.match_like(b.dict, b.entry_off, p, null_text=null)
                assert flags[b.values[k]].cpu().tolist() == [M.like(s, p) for s in tx]
            rank, found = ctx.find_strings(b.dict, b.entry_off, [b"alpha", b"beta", b"zz"])
            assert rank.cpu().tolist() == [bisect.bisect_left(ents, q) for q in (b"alpha", b"beta", b"zz")]
            assert found.cpu().tolist() == [q in ents for q in (b"alpha", b"beta", b"zz")]


def test_filter_write_read_round_trip(tmp_path):
    """like and between filter a table; write_table and read_table give back exactly the host-filtered rows."""
    from zdw_b200 import ColumnTable, between, like, read_table, write_table
    image = O.golden("analytics-hits.zdw")
    sch, _, _ = O.read_header(image)
    hdr, t = read_table(image)
    dt = next(k for k, c in enumerate(t.columns) if hdr.types[c] == DATETIME)
    txt = next(k for k, c in enumerate(t.columns) if hdr.types[c] in TEXT_LIKE and hdr.types[c] not in (DATETIME, DECIMAL)
               and len(set(t.values[k].tolist())) > 5)
    s_dt, s_txt = t.strings(dt), t.strings(txt)
    mid = sorted(set(x for x in s_dt if x))[len(set(s_dt)) // 2]
    some = next(x for x in s_txt if x and len(x) >= 2)
    pat = b"%" + esc(some[:2]) + b"%"
    keep = like(hdr, t, txt, pat) & between(hdr, t, dt, b"", mid)
    want = [i for i in range(len(s_dt)) if M.like(s_txt[i] or b"", pat) and (s_dt[i] or b"") <= mid]
    assert keep.nonzero().flatten().tolist() == want and 0 < len(want) < len(s_dt)
    path = tmp_path / "f.zdw"
    write_table(path, hdr, ColumnTable(t.values[:, keep], t.dicts, t.columns, [int(keep.sum())]))
    _, back = read_table(path)
    for k, c in enumerate(t.columns):
        if t.dicts[k] is None:
            assert back.values[k].tolist() == t.values[k][keep].tolist()
        else:
            full = t.strings(k)
            assert back.strings(k) == [full[i] for i in want]


def test_predicates_wait_for_torchs_stream(ctx):
    """The codes are produced on torch's current stream behind a spin kernel: the predicates must see the final codes.
    Context.find_strings on its own must not wait for that stream."""
    import torch
    from zdw_b200 import ColumnTable, between, isin, like
    from test_gpu_columns import MIXED, _mixed_tsv
    sch = O.parse_desc(corpus.desc(MIXED))
    r = O.encode(sch, _mixed_tsv(3000, 9), rows_per_block=1000)
    hdr, t, texts = host_table(r.data)
    k = next(k for k, c in enumerate(t.columns) if hdr.types[c] == 0)
    d, eo = t.dicts[k]
    zeros = torch.zeros_like(t.values)
    late = torch.empty_like(t.values)
    torch.add(zeros, t.values, out=late)
    late.fill_(-1)
    warm = like(hdr, t, k, b"%a%"), isin(hdr, t, k, [b"beta"]), between(hdr, t, k, b"a", b"c"), ctx.find_strings(d, eo, [b"x"])
    del warm
    torch.cuda.synchronize()
    torch.cuda._sleep(4_000_000_000)
    rank, found = ctx.find_strings(d, eo, [b"alpha", b"beta", b"gamma1"])
    assert not torch.cuda.current_stream().query(), "find_strings waited for torch's stream"
    torch.add(zeros, t.values, out=late)  # queued behind the spin
    tl = ColumnTable(late, t.dicts, t.columns, t.block_rows)
    tx = texts[k]
    ents = entries(bytes(d.cpu().numpy().tobytes()), eo.cpu().tolist())
    assert rank.cpu().tolist() == [bisect.bisect_left(ents, q) for q in (b"alpha", b"beta", b"gamma1")]
    assert like(hdr, tl, k, b"%a%").cpu().tolist() == [M.like(s, b"%a%") for s in tx]
    assert isin(hdr, tl, k, [b"beta", b""]).cpu().tolist() == [s in (b"beta", b"") for s in tx]
    assert between(hdr, tl, k, b"a", b"c").cpu().tolist() == [b"a" <= s <= b"c" for s in tx]


def test_null_cells_take_the_null_flag():
    """Code -1 takes the flag of the column's null text: "" for text, "0.000000000000" for DECIMAL."""
    from zdw_b200 import between, isin, like
    from test_gpu_columns import MIXED, _mixed_tsv
    sch = O.parse_desc(corpus.desc(MIXED))
    r = O.encode(sch, _mixed_tsv(500, 3))
    hdr, t, texts = host_table(r.data)
    with_null = 0
    for k, c in enumerate(t.columns):
        codes = t.values[k].cpu().tolist()
        if -1 not in codes:
            continue
        with_null += hdr.types[c]
        null = b"0.000000000000" if hdr.types[c] == DECIMAL else b""
        nulls = [i for i, v in enumerate(codes) if v == -1]
        for p, want in ((b"", null == b""), (b"0.0%", null != b""), (b"%", True), (b"_%", null != b"")):
            got = like(hdr, t, k, p).cpu().tolist()
            assert all(got[i] == want for i in nulls), (k, p)
        assert all(isin(hdr, t, k, [null]).cpu().tolist()[i] for i in nulls)
        assert not any(isin(hdr, t, k, [b"zz"]).cpu().tolist()[i] for i in nulls)
        assert all(between(hdr, t, k, null, null).cpu().tolist()[i] for i in nulls)
    assert with_null >= DECIMAL + 1  # a DECIMAL column and a text one had -1 cells
    from zdw_b200 import read_table
    h2, t2 = read_table(r.data, ["a", "b"])
    with pytest.raises(ValueError):
        like(h2, t2, 0, b"%")
    with pytest.raises(ValueError):
        isin(h2, t2, 0, [b"x"])
    with pytest.raises(ValueError):
        between(h2, t2, 0, b"a", b"b")
