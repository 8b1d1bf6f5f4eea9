"""GPU tests of the merged dictionaries (zdwb_merge_codes, read_table).  The oracle is the C restatement's decoded text
(or hand-built parts) and Python's sorted(set(...)).  Every check covers three things: the merged dictionary is strictly
increasing and dense; it equals the sorted set of the strings the codes stand for; and every cell rendered with it
gives the expected text."""
import ctypes as C
import gzip
import lzma
import random

import pytest

import corpus
import gpuutil as G
import oracle as O
from columns_util import TEXT_LIKE, entries, render
from test_gpu_columns import MIXED, _mixed_tsv

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from zdw_b200 import Context
    c = Context(0)
    yield c
    c.close()


def merged_entries(dct, eo, codes):
    """The merged dictionary's entries, after checking that it is strictly increasing and dense for `codes`."""
    d = bytes(dct.cpu().numpy().tobytes())
    offs = eo.cpu().tolist()
    assert offs[-1] == len(d)
    if not d:
        assert offs == [0]
        assert all(c == -1 for c in codes)
        return []
    assert d[:1] == b"\0" and all(d[b - 1] == 0 for b in offs[1:])
    ents = entries(d, offs)
    assert all(a < b for a, b in zip(ents, ents[1:])), "merged entries not strictly increasing"
    assert set(c for c in codes if c >= 0) == set(range(len(ents))), "merged codes not dense"
    return ents


def check_merged(m, want):
    """m: MergedCodes; want: the string (or None) of every code, parts in order."""
    codes = m.codes.cpu().tolist()
    assert len(codes) == len(want)
    ents = merged_entries(m.dict, m.entry_off, codes)
    assert ents == sorted(set(w for w in want if w is not None))
    assert [None if c < 0 else ents[c] for c in codes] == want


def mk_part(ents, codes):
    """A part on the device: a dictionary of `ents` (laid out as a block's) and `codes` into it."""
    import torch
    d = b"\0" + b"".join(e + b"\0" for e in ents)
    eo, at = [], 1
    for e in ents:
        eo.append(at)
        at += len(e) + 1
    eo.append(at)
    dt = torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda() if ents else torch.empty(0, dtype=torch.uint8, device="cuda")
    return (dt, torch.tensor(eo if ents else [], dtype=torch.int64, device="cuda"),
            torch.tensor(codes, dtype=torch.int64, device="cuda"))


def merge_host_parts(ctx, spec):
    """spec: [(sorted distinct entries, codes)]; merges them and checks the result."""
    import torch
    parts = [mk_part(e, c) for e, c in spec]
    torch.cuda.synchronize()
    m = ctx.merge_codes(parts)
    want = [None if c < 0 else e[c] for e, cs in spec for c in cs]
    check_merged(m, want)
    return m


# ----------------------------------------------------------------------------- read_table against the C restatement

def check_table(image, names, rows_per_block=None, path=None):
    """read_table of the file (or of `path`) against the C restatement's decode of the same columns."""
    from zdw_b200 import read_columns, read_table
    sch, _, _ = O.read_header(image)
    cols = [sch.names.index(n) for n in names]
    hdr, t = read_table(path if path is not None else image, names)
    assert t.columns == cols and hdr.names == sch.names
    ocol = [-1] * sch.ncols
    for k, c in enumerate(cols):
        ocol[c] = k
    want = O.decode(image, out_col=ocol, n_out=len(cols))
    assert want.rc == 0
    assert tuple(t.values.shape) == (len(cols), want.total_rows) and sum(t.block_rows) == want.total_rows
    V = t.values.cpu().tolist()
    rendered = []
    for k, c in enumerate(cols):
        typ = sch.types[c]
        if typ in TEXT_LIKE:
            dct, eo = t.dicts[k]
            ents = merged_entries(dct, eo, V[k])
            strs = [ents[v] for v in V[k] if v >= 0]
            assert ents == sorted(set(strs))
            assert t.strings(k) == [None if v < 0 else ents[v] for v in V[k]]
        else:
            assert t.dicts[k] is None
            ents = []
        rendered.append([render(typ, v, ents) for v in V[k]])
    got = b"".join(b"\t".join(row) + b"\n" for row in zip(*rendered)) if rendered and V[0] else b""
    assert got == want.tsv, G.first_diff(got, want.tsv)
    # the non-text rows are the blocks' rows concatenated
    _, blocks = read_columns(image, names)
    assert len(blocks) == len(t.block_rows) and [b.nrows for b in blocks] == t.block_rows
    if rows_per_block:
        assert all(n <= rows_per_block for n in t.block_rows)
    import torch
    for k, c in enumerate(cols):
        if sch.types[c] not in TEXT_LIKE:
            assert torch.equal(t.values[k], torch.cat([b.values[k] for b in blocks]))
    return t


@pytest.mark.parametrize("rows_per_block", [1, 7, 1000])
def test_read_table_mixed(tmp_path, rows_per_block):
    sch = O.parse_desc(corpus.desc(MIXED))
    r = O.encode(sch, _mixed_tsv(1500 if rows_per_block > 1 else 40, 3), rows_per_block=rows_per_block)
    assert r.rc == 0 and r.nblocks > 1
    rng = random.Random(rows_per_block)
    for suffix, data in (("", r.data), (".gz", gzip.compress(r.data)), (".xz", lzma.compress(r.data))):
        names = rng.sample(sch.names, rng.randint(1, len(sch.names)))
        p = tmp_path / f"f.zdw{suffix}"
        p.write_bytes(data)
        check_table(r.data, names, rows_per_block, path=p)
    check_table(r.data, list(sch.names), rows_per_block)


CASES = {c[0]: c for c in corpus.cases() if "expect_rc" not in c[3]}
CORPUS = [n for n in CASES if n.startswith(("d7_text_like", "d9_dict", "d14_long_common_prefixes", "mixed_3000", "d1"))]


@pytest.mark.parametrize("name", CORPUS)
def test_corpus_in_blocks_of_100(name):
    _, desc, tsv, opts = CASES[name]
    sch = O.parse_desc(desc)
    r = O.encode(sch, tsv, trim=bool(opts.get("trim")), rows_per_block=100)
    if r.rc != 0 or r.total_rows == 0:
        return
    check_table(r.data, list(sch.names), 100)


def _golden_reencoded(name, rows_per_block):
    sch = O.parse_desc(O.golden(f"{name}.desc.sql"))
    r = O.encode(sch, O.golden(f"{name}.sql"), rows_per_block=rows_per_block)
    assert r.rc == 0 and r.nblocks > 1
    return sch, r


def test_golden_movie_tickets_in_blocks():
    """About half a million distinct titles, almost none shared across blocks: every merge level does real work."""
    sch, r = _golden_reencoded("movie_tickets", 60000)
    assert r.nblocks >= 8
    t = check_table(r.data, list(sch.names))
    assert max(int(e.numel()) for e in (d[1] for d in t.dicts if d is not None)) > 100000


def test_golden_analytics_hits_in_blocks():
    """Low cardinality, heavy sharing across blocks."""
    sch, r = _golden_reencoded("analytics-hits", 300)
    rng = random.Random(9)
    text = [n for n, ty in zip(sch.names, sch.types) if ty in TEXT_LIKE]
    names = rng.sample(text, 12) + rng.sample(sch.names, 12)
    check_table(r.data, list(dict.fromkeys(names)))


# ----------------------------------------------------------------------------- part shapes

def _strs(rng, n, alphabet=b"abc", maxlen=4):
    out = set()
    while len(out) < n:
        out.add(bytes(rng.choice(alphabet) for _ in range(rng.randint(0, maxlen))))
    return sorted(out)


@pytest.mark.parametrize("P", [1, 2, 3, 5, 17, 215])
def test_part_counts(ctx, P):
    rng = random.Random(P)
    spec = []
    for p in range(P):
        ents = _strs(rng, rng.randint(1, 40), b"abcdefgh", 6)
        spec.append((ents, [rng.randrange(-1, len(ents)) for _ in range(rng.randint(0, 60))]))
    merge_host_parts(ctx, spec)


def test_degenerate_parts(ctx):
    ents = [b"a", b"b", b"c"]
    shapes = [
        [(ents, [])],                                   # n = 0
        [(ents, [-1, -1, -1])],                         # all codes -1
        [([], [])],                                     # entries = 0, NULL dict
        [([], [-1, -1])],
        [(ents, []), ([], [-1]), (ents, [-1, 2]), (ents, []), ([b"c", b"d"], [1, 0, 1])],
        [(ents, [1]), (ents, [-1]), ([], [])],          # entries but no referenced entry in the later parts
        [],                                             # no parts at all
        [(ents, [-1])] * 999 + [(ents, [1, 2])],        # far more parts than references
    ]
    for spec in shapes:
        merge_host_parts(ctx, spec)


def test_identical_disjoint_and_prefix_chains(ctx):
    ents = [b"apple", b"banana", b"cherry", b"date"]
    merge_host_parts(ctx, [(ents, [0, 1, 2, 3, 3])] * 6)                        # identical parts
    evens = [b"%03d" % i for i in range(0, 200, 2)]
    odds = [b"%03d" % i for i in range(1, 200, 2)]
    merge_host_parts(ctx, [(evens, list(range(100))), (odds, list(range(100))), (evens, [5, 7])])  # interleaved
    chain = [b"a" * k for k in range(1, 40)] + [b"ab" * k for k in range(1, 30)]
    spec = []
    for p in range(7):
        sub = sorted(set(chain[p::7] + chain[(p + 3) % 7::7]))
        spec.append((sub, list(range(len(sub)))[::-1]))
    merge_host_parts(ctx, spec)                                                    # prefix chains across parts


def test_strings_that_differ_past_the_prefix_key(ctx):
    rng = random.Random(3)
    spec = []
    for p in range(9):
        ents = set()
        for L in (1, 2, 15, 16, 17, 31, 32, 33, 64, 100, 255, 300):
            base = bytes([0x61 + (p % 3)]) * (L - 1)
            for last in (0x01, 0x7F, 0x80, 0xFF, rng.randint(1, 255)):
                ents.add(base + bytes([last]))
        ents = sorted(ents)
        spec.append((ents, [rng.randrange(-1, len(ents)) for _ in range(200)]))
    merge_host_parts(ctx, spec)
    high = sorted({bytes([b]) * k for b in (0x01, 0x7F, 0x80, 0xFF) for k in (1, 16, 17, 40)})
    merge_host_parts(ctx, [(high, list(range(len(high)))), (high[::2], list(range(len(high[::2]))))])


def test_emit_copies_long_entries_in_chunks_and_in_bytes(ctx):
    """k_merge_emit copies an entry of 64 bytes or more in 16-byte chunks when its source and destination share their
    address mod 16, and byte by byte otherwise.  Both paths are forced here: the input dictionaries are torch
    allocations (512-byte aligned) and the output dictionary an arena piece (256-byte aligned), so the offsets decide.
    The one referenced entry sits at input offset 1 + pad and goes to output offset 1: pad = 0, 16, 32 take the chunks
    (after a 15-byte head), the other pads the bytes."""
    import torch
    for L in (63, 64, 65, 79, 80, 81, 300, 1000):
        s = bytes((7 * i + L) % 255 + 1 for i in range(L))
        for pad in (0, 1, 15, 16, 17, 32):
            if pad == 0:
                d, eo = b"\0" + s + b"\0", [1, L + 2]
            else:  # an unreferenced entry of pad - 1 bytes in front
                d, eo = b"\0" + b"\x01" * (pad - 1) + b"\0" + s + b"\0", [1, 1 + pad, 1 + pad + L + 1]
            code = len(eo) - 2
            part = (torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda(), torch.tensor(eo, dtype=torch.int64).cuda(),
                    torch.tensor([code, -1, code], dtype=torch.int64).cuda())
            assert part[0].data_ptr() % 16 == 0
            torch.cuda.synchronize()
            check_merged(ctx.merge_codes([part]), [s, None, s])
        # several long entries: the later ones land at other output alignments
        ents = sorted({bytes([c]) * k + s for c in (2, 3, 4, 5) for k in range(1, 5)})
        merge_host_parts(ctx, [(ents, list(range(len(ents)))), (ents[::3], [0, 1, 2])])


def test_random_part_sets(ctx):
    rng = random.Random(2024)
    for case in range(300):
        P = rng.randint(1, 12)
        spec = []
        for p in range(P):
            ents = _strs(rng, rng.randint(0, 12), b"ab\x01\xff", rng.choice([3, 20]))
            n = rng.randint(0, 30)
            spec.append((ents, [rng.randrange(-1, len(ents)) if ents else -1 for _ in range(n)]))
        merge_host_parts(ctx, spec)


def test_two_columns_and_two_files_share_a_dictionary(ctx):
    from zdw_b200 import read_columns
    sch = O.parse_desc(corpus.desc(MIXED))
    r1 = O.encode(sch, _mixed_tsv(900, 21), rows_per_block=100)
    r2 = O.encode(sch, _mixed_tsv(700, 22), rows_per_block=64)
    _, b1 = read_columns(r1.data, ["b", "d", "j"])
    _, b2 = read_columns(r2.data, ["b"])
    parts = [(b.dict, b.entry_off, b.values[0]) for b in b1] + [(b.dict, b.entry_off, b.values[1]) for b in b1]
    want = [s for b in b1 for s in b.strings(0)] + [s for b in b1 for s in b.strings(1)]
    m = ctx.merge_codes(parts)
    check_merged(m, want)
    parts = [(b.dict, b.entry_off, b.values[0]) for b in b1] + [(b.dict, b.entry_off, b.values[0]) for b in b2]
    want = [s for b in b1 for s in b.strings(0)] + [s for b in b2 for s in b.strings(0)]
    m = ctx.merge_codes(parts)
    check_merged(m, want)
    codes = m.codes.cpu().tolist()
    first = {}
    for c, s in zip(codes, want):  # equal codes iff equal strings
        assert first.setdefault(s, c) == c
    # a column a block does not use: all -1, its part references nothing
    check_merged(ctx.merge_codes([(b.dict, b.entry_off, b.values[2]) for b in b1]), [None] * 900)


def test_c4_four_blocks_every_used_text_column(ctx):
    import bench
    synth = bench.Synth()
    types = synth.schema.types
    n_rows = 32768
    cap = synth.cap_for(n_rows)
    buf = (C.c_uint8 * cap)()
    blocks = []
    for b in range(4):
        n = synth.block_into(b, n_rows, C.addressof(buf), cap)
        blocks.append(ctx.encode_block(types, bytes((C.c_uint8 * n).from_address(C.addressof(buf)))).data)
    probe = ctx.decode_columns(types, blocks[0], list(range(len(types))))
    text = [c for c in range(len(types)) if types[c] in TEXT_LIKE]
    cbs = [ctx.decode_columns(types, z, text) for z in blocks]
    import torch
    used = [k for k in range(len(text)) if int(torch.stack([cb.values[k].max() for cb in cbs]).max()) >= 0]
    assert len(used) > 10 and probe.nrows == n_rows
    dicts = [entries(bytes(cb.dict.cpu().numpy().tobytes()), cb.entry_off.cpu().tolist()) for cb in cbs]
    vals = [cb.values.cpu().tolist() for cb in cbs]
    for k in used:
        m = ctx.merge_codes([(cb.dict, cb.entry_off, cb.values[k]) for cb in cbs])
        check_merged(m, [None if v < 0 else ents[v] for ents, V in zip(dicts, vals) for v in V[k]])


# ----------------------------------------------------------------------------- errors

def test_errors_and_recovery(ctx):
    import torch
    from zdw_b200 import ZdwError, capi
    good = mk_part([b"a", b"b"], [0, 1])

    def fails(parts, code):
        torch.cuda.synchronize()
        with pytest.raises(ZdwError) as ei:
            ctx.merge_codes(parts)
        assert ei.value.code == code, ei.value

    # n_parts > 0 with NULL parts; a part with n > 0 and NULL codes
    out = capi._MergeOut()
    assert ctx._L.zdwb_merge_codes(ctx._h, None, 2, C.byref(out)) == 4
    arr = (capi._CodePart * 1)(capi._CodePart(good[0].data_ptr(), good[1].data_ptr(), 2, good[0].numel(), None, 5))
    assert ctx._L.zdwb_merge_codes(ctx._h, arr, 1, C.byref(out)) == 4
    # codes < -1 or >= entries
    fails([good, mk_part([b"a"], [0, -2])], 4)
    fails([mk_part([b"a", b"b"], [2]), good], 4)
    fails([mk_part([], [0])], 4)
    # bad offsets of a referenced entry: not increasing, past dict_bytes
    d, eo, c = mk_part([b"a", b"b", b"c"], [1])
    for bad in ([1, 3, 3, 7], [1, 3, 99, 7], [1, 5, 3, 7]):
        fails([good, (d, torch.tensor(bad, dtype=torch.int64, device="cuda"), c)], 4)
    # the same offsets are fine when no code references the entry
    ok = merge_host_parts(ctx, [([b"a", b"b", b"c"], [0])])
    assert ok.entries == 1
    torch.cuda.synchronize()
    check_merged(ctx.merge_codes([(d, torch.tensor([1, 3, 5, 99], dtype=torch.int64, device="cuda"),
                                   torch.tensor([0, 1], dtype=torch.int64, device="cuda"))]), [b"a", b"b"])
    # referenced entries not strictly increasing (equal, descending, past the prefix key)
    fails([mk_part([b"b", b"a"], [0, 1])], 4)
    fails([good, mk_part([b"a", b"a"], [0, 1])], 4)
    fails([mk_part([b"x" * 20 + b"b", b"x" * 20 + b"a"], [1, 0])], 4)
    merge_host_parts(ctx, [([b"b", b"a"], [1])])  # an unsorted pair is fine when one of them is not referenced
    # more referenced entries than supported
    ctx.set_tuning("merge_max_refs", 2)
    try:
        fails([mk_part([b"a", b"b", b"c"], [0, 1, 2])], 5)
        merge_host_parts(ctx, [([b"a", b"b", b"c"], [0, 2, 2])])
    finally:
        ctx.set_tuning("merge_max_refs", 1 << 32)
    # the context still works: a merge, and a block decoded to rows and columns
    merge_host_parts(ctx, [([b"a", b"b"], [0, 1]), ([b"b", b"c"], [1, 0])])
    one = O.parse_desc(corpus.desc([("a", "varchar(9)"), ("b", "int(11)")]))
    img = O.encode(one, b"hello\t1\nworld\t2\n").data
    _, _, hl = O.read_header(img)
    assert ctx.decode_block(one.types, img[hl:]).tsv == b"hello\t1\nworld\t2\n"
    assert ctx.decode_columns(one.types, img[hl:], [0]).strings(0) == [b"hello", b"world"]


def test_outputs_survive_work_queued_on_torchs_stream(ctx):
    """The outputs are copied out before the context's next call re-uses its memory, even while torch's current stream
    is busy: a spin kernel holds that stream while 40 merges run (warmed up first, so that no allocation synchronises
    the device)."""
    import torch
    rng = random.Random(77)
    specs = []
    for i in range(40):
        spec = []
        for p in range(rng.randint(2, 6)):
            ents = _strs(rng, rng.randint(1, 30), b"abcdef", 5)
            spec.append((ents, [rng.randrange(-1, len(ents)) for _ in range(500)]))
        specs.append(spec)
    parts = [[mk_part(e, c) for e, c in spec] for spec in specs]
    torch.cuda.synchronize()
    warm = [ctx.merge_codes(p) for p in parts]
    del warm
    torch.cuda.synchronize()
    torch.cuda._sleep(4_000_000_000)
    results = [ctx.merge_codes(p) for p in parts]
    assert not torch.cuda.current_stream().query(), "the spin ended before the merges ran: nothing was tested"
    for m, spec in zip(results, specs):
        check_merged(m, [None if c < 0 else e[c] for e, cs in spec for c in cs])
