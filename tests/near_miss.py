"""Seeded near-miss inputs for the two places that skip work on "same as the row before".

The row-delta pass 1 (k_pass1d) gives a field no record when its bytes equal the same column of the row before; the
delta row writer (k_dec_write_delta) copies a decoded row's unchanged stretches from the row before and renders only the
changed items.  A wrong verdict or a wrong source offset in either gives a valid file or plausible text that is wrong,
and random data hides it: a field drawn afresh differs at byte 0, and a neighbouring column's value differs anyway.
These families are built so that the only thing between a right and a wrong answer is the decision under test.

Every family is a tuple (name, desc, tsv, canonical, claims):
- canonical: decoding the file gives back the source bytes up to the last newline (`expected_tsv`: an unterminated
  last line is no row, as in the reference's reader).  Such families have no empty integer cells and spell every
  number canonically.
- claims: a dict of what the family is built to hit, as lists of tuples whose second element is a row index of `tsv`
  (tests/test_near_miss_host.py checks every one of them on the text), plus "opts": the encode options (trim,
  rows_per_block) the family must be encoded with.

Encode families (E*), each placed three ways: as a file under 64 KiB (the compares' clamped loads), in the middle of a
file over 256 KiB (the unclamped ones: more than 64 KiB + 32 bytes in front of the end), as the last rows of the buffer
with the differing byte its last byte: once in front of the final newline, once without one (then that last line is
dropped, and the rows in front of it are parsed and compared right up to the buffer's end).  Decode families (D*) are canonical.
Changed bytes never become a tab, a newline, a backslash or NUL.
"""
from __future__ import annotations

import random
from functools import lru_cache

import corpus

BAD = frozenset(b"\t\n\\\0")
ALPHA = b"abcdefghijklmnopqrstuvwxy0123456789ABCDEFGHIJKLMNOP"  # +1, ^0x01 and ^0x80 of these are never BAD
SMALL_MAX = 60 * 1024   # a "small" file: under 64 KiB, so no compare takes the unclamped loads
PAD = 128 * 1024        # filler in front of and behind a "mid" placement


def _txt(rng, n):
    return bytes(rng.choices(ALPHA, k=n))


def _join(rows, final_newline=True):
    t = b"\n".join(rows)
    return t + b"\n" if final_newline and rows else t


def expected_tsv(tsv: bytes) -> bytes:
    """what decoding a canonical family's file gives: the source up to its last newline"""
    return tsv[:tsv.rfind(b"\n") + 1]


def _sub(claims, s, e, shift=0):
    """claims of rows s .. e - 1 whose row before is in the range too, renumbered from s (plus shift)."""
    return [(c[0], c[1] - s + shift) + tuple(c[2:]) for c in claims if s < c[1] < e]


def _chunks(rows, limit):
    """runs of consecutive rows under `limit` bytes as a file; each run starts with the last row of the run before,
    so that every pair of neighbouring rows is in some run"""
    out, s = [], 0
    while True:
        size, e = 0, s
        while e < len(rows) and (e < s + 2 or size + len(rows[e]) + 1 <= limit):
            size += len(rows[e]) + 1
            e += 1
        out.append((s, e))
        if e >= len(rows):
            return out
        s = e - 1


def _place(name, desc, rows, claims, pad_rows, tail, tail_claims):
    """The three placements of an encode family.  tail: rows that end the "end" placement (their last changed field
    ends the buffer), with claims numbered from the tail's first row."""
    out = []
    chunks = _chunks(rows, SMALL_MAX)
    for i, (s, e) in enumerate(chunks):
        out.append((f"{name}/small{i}", desc, _join(rows[s:e]), True, _group(_sub(claims, s, e))))
    # mid: filler in front and behind, more than 64 KiB + 32 bytes of it behind the last row of the family
    front, back, n = [], [], 0
    while n < PAD:
        front.append(pad_rows(len(front)))
        n += len(front[-1]) + 1
    n = 0
    while n < PAD:
        back.append(pad_rows(len(front) + len(back) + 7))
        n += len(back[-1]) + 1
    mid = front + rows + back
    out.append((f"{name}/mid", desc, _join(mid), True, _group(_sub(claims, 0, len(rows), len(front)))))
    # end: the last run of rows under 64 KiB (less the tail), then the tail
    tail_len = sum(len(r) + 1 for r in tail)
    s, e = _chunks(rows, max(SMALL_MAX - tail_len, 1))[-1]
    end = rows[s:e] + tail
    cl = _sub(claims, s, e) + [(c[0], c[1] + e - s) + tuple(c[2:]) for c in tail_claims]
    for nl in (True, False):
        out.append((f"{name}/end{'_nl' if nl else ''}", desc, _join(end, nl), True, _group(cl)))
    return out


def _group(claims):
    g = {}
    for c in claims:
        g.setdefault(c[0], []).append(c[1:])
    return g


# ----------------------------------------------------------------------------------------------- E1: one byte off

E1_LENGTHS = list(range(1, 21)) + [31, 32, 33, 47, 48, 49, 63, 64, 65, 127, 128, 129, 130, 255, 256, 257, 1000, 4000]
E1_CHANGES = (("inc", lambda b: b + 1), ("x01", lambda b: b ^ 0x01), ("x80", lambda b: b ^ 0x80))
E1_DESC = corpus.desc([("pre", "varchar(255)"), ("k", "int(11)"), ("f", "text")])
E1_COL = 2


def e1_offsets(L):
    return sorted({o for o in (0, 1, 2, 3, 4, 5, 7, 8, 11, 12, 15, 16, 17, L // 2, L - 5, L - 4, L - 3, L - 2, L - 1)
                   if 0 <= o < L})


def _poke(v, off, fn):
    nb = fn(v[off])
    assert nb not in BAD and nb != v[off]
    return v[:off] + bytes([nb]) + v[off + 1:]


def _e1_rows(L):
    """Units of four rows: base, one byte off, base again, an exact repeat.  The varchar in front of the field takes
    lengths 0-19 at random, so that the field and its copy in the row before meet at every alignment."""
    rng = random.Random(1000 + L)
    base = _txt(rng, L)
    rows, claims = [], []

    def row(u, role, v):
        rows.append(b"\t".join([_txt(rng, rng.randrange(20)), b"%d" % (1000 + len(rows)), v]))

    u = 0
    while u < 64:  # (short fields have few offsets: their units repeat until the alignments are all there)
        for off in e1_offsets(L):
            for _, fn in E1_CHANGES:
                r = len(rows)
                row(u, 0, base)
                row(u, 1, _poke(base, off, fn))
                row(u, 2, base)
                row(u, 3, base)
                claims += [("one_off", r + 1, E1_COL, L, off), ("one_off", r + 2, E1_COL, L, off), ("repeat", r + 3, E1_COL)]
                u += 1
    return rows, claims, base


def _e1_pad(rng):
    return lambda i: b"\t".join([_txt(rng, i % 13), b"%d" % (5 + i), _txt(rng, 150 + i % 97)])


@lru_cache(maxsize=None)
def e1_families():
    out = []
    for L in E1_LENGTHS:
        rows, claims, base = _e1_rows(L)
        tail = [b"\t".join([b"tail", b"1", base]), b"\t".join([b"tai", b"2", _poke(base, L - 1, E1_CHANGES[2][1])])]
        out += _place(f"E1_L{L}", E1_DESC, rows, claims, _e1_pad(random.Random(L)), tail,
                      [("one_off", 1, E1_COL, L, L - 1)])
    # a block cut between a base row and its one-off row: 41 = 4 * 10 + 1 rows per block (unit 10's one-off row opens
    # block 1)
    rows, claims, _ = _e1_rows(17)
    out.append(("E1_L17/rows_per_block41", E1_DESC, _join(rows), True, {**_group(claims), "opts": {"rows_per_block": 41}}))
    return out


# ------------------------------------------------------------------------------------------ E2: neighbour-equal

E2_NCOLS = 4096
E2_FOCUS = [(0, 1), (31, 32), (63, 64), (1023, 1024), (4094, 4095)]
E2_LENGTHS = [1, 4, 16, 17, 40, 129]
E2_DESC = corpus.desc([(f"c{i}", "text") for i in range(E2_NCOLS)])
DCAP = 280  # non-empty fields of a row the row-delta pass 1 holds


def _e2_rows(L):
    """Row r, column c holds g(c - r) in "left" segments and g(c + r) in "right" ones: the value of the row before in
    column c - 1 (c + 1), of the same length, and one more or less than its own column's value there (so the two differ
    late, in the decimal counter that ends the value).  The focus pairs are filled in every row; the other filled
    columns are drawn afresh per row, so the rank of a column in the bitmap shifts from row to row."""
    rng = random.Random(2000 + L)
    prefix = _txt(rng, max(L - 10, 0))

    def g(x):
        return (prefix + b"%010d" % (x + 10 ** 6))[-L:] if L >= 10 else (b"%010d" % (x + 10 ** 6))[-L:]

    budget = {1: DCAP, 4: 250, 16: 200, 17: 180, 40: 100, 129: 40}[L]
    focus = sorted({c for p in E2_FOCUS for c in p})
    rows, claims, sets = [], [], []
    nrows = 18
    for r in range(nrows):
        s = 1 if (r // 6) % 2 == 0 else -1  # segments of six rows: left, right, left
        want = budget if r % 3 == 0 else rng.randrange(budget // 2, budget + 1)
        filled = set(focus) | {c for a, b in E2_FOCUS for c in range(max(a - 6, 0), min(b + 7, E2_NCOLS))
                               if rng.random() < 0.5}  # the columns around a focus pair go empty or filled
        extra = sorted(filled - set(focus))
        rng.shuffle(extra)
        while len(filled) > want:
            filled.discard(extra.pop())
        while len(filled) < want:
            filled.add(rng.randrange(E2_NCOLS))
        filled = sorted(filled)
        cells = [b""] * E2_NCOLS
        for c in filled:
            cells[c] = g(c - s * r)
        rows.append(b"\t".join(cells))
        fs = set(filled)
        if r and (r // 6) == ((r - 1) // 6):
            prev = sets[-1]
            for c in filled:
                nc = c - s
                if 0 <= nc < E2_NCOLS and nc in prev:
                    claims.append(("neighbour", r, c, nc))
        sets.append(fs)
    # the last row's column 4095 is one more or less than in the row before: it differs in its last byte
    claims.append(("last_byte", nrows - 1, E2_NCOLS - 1))
    return rows, claims


def _e2_pad(rng):
    def row(i):
        cells = [b""] * E2_NCOLS
        for c in rng.sample(range(E2_NCOLS), 12):
            cells[c] = _txt(rng, 3 + (c + i) % 40)
        return b"\t".join(cells)
    return row


@lru_cache(maxsize=None)
def e2_families():
    out = []
    for L in E2_LENGTHS:
        rows, claims = _e2_rows(L)
        out += _place(f"E2_L{L}", E2_DESC, rows, claims, _e2_pad(random.Random(L)), [], [])
    return out


# --------------------------------------------------------------------------------- E3: same value, other bytes

E3_INT_DESC = corpus.desc([("a", "int(11)"), ("b", "bigint(20)"), ("c", "bigint(20) unsigned"), ("t", "text")])
E3_INT_GROUPS = [[b"7", b"07", b"+7", b"7", b"07", b"7"], [b"0", b"-0", b"00", b"0", b"-0", b"+0", b"0"],
                 [b"18446744073709551615", b"18446744073709551616", b"18446744073709551617", b"18446744073709551616"],
                 [b"-18446744073709551616", b"-18446744073709551615", b"-18446744073709551616"],
                 [b"184467440737095516150", b"184467440737095516151", b"184467440737095516150"],
                 [b"9223372036854775807", b"9223372036854775808", b"9223372036854775809", b"9223372036854775808"],
                 [b"99999999999", b"99999999998", b"99999999999"],
                 [b"00000000000000000000001", b"+0000000000000000000001", b"00000000000000000000001"]]
E3_TXT_DESC = corpus.desc([("t", "text"), ("u", "varchar(255)"), ("k", "int(11)")])


def _e3_txt_groups():
    rng = random.Random(3)
    x16, x128, x15 = _txt(rng, 16), _txt(rng, 128), _txt(rng, 15)
    return [[b"abc", b"abc ", b"abc  ", b"abc", b"abc  "], [b"abc ", b"abcd", b"abc "],
            [x16, x16 + b" ", x16, x16 + b"  "], [x15 + b" ", x15 + b"z", x15 + b" "],
            [x128, x128 + b" ", x128, x128 + b"   "], [x128[:-1] + b" ", x128, x128[:-1] + b" "],
            [b" ", b"  ", b""]]


@lru_cache(maxsize=None)
def e3_families():
    out = []
    rs, cl = [], []
    for grp in E3_INT_GROUPS:
        for i, v in enumerate(grp):
            rs.append(b"\t".join([v, v, v, b"r%d" % len(rs)]))
            if i:
                cl.append(("same_spelling_len" if len(v) == len(grp[i - 1]) else "other_len", len(rs) - 1, 0))
    rt, ct = [], []
    for grp in _e3_txt_groups():
        for i, v in enumerate(grp):
            rt.append(b"\t".join([v, v, b"%d" % len(rt)]))
            if i:
                ct.append(("trimmed_equal" if v.rstrip(b" ") == grp[i - 1].rstrip(b" ") else "trimmed_differ", len(rt) - 1, 0))
    rng = random.Random(33)
    for name, desc, rows, claims, trim, pad in (("E3_int", E3_INT_DESC, rs, cl, False,
                                                 lambda i: b"\t".join([b"%d" % (i % 90 + 1)] * 3 + [_txt(rng, 200)])),
                                                ("E3_trim", E3_TXT_DESC, rt, ct, True,
                                                 lambda i: b"\t".join([_txt(rng, 150), _txt(rng, 50) + b" ", b"%d" % i]))):
        opts = {"opts": {"trim": trim}}
        out.append((f"{name}/small", desc, _join(rows), False, {**_group(claims), **opts}))
        front = [pad(i) for i in range(PAD // 200)]
        back = [pad(i + 5000) for i in range(PAD // 200)]
        out.append((f"{name}/mid", desc, _join(front + rows + back), False,
                    {**_group(_sub(claims, 0, len(rows), len(front))), **opts}))
    return out


def encode_families():
    return e1_families() + e2_families() + e3_families()


# ------------------------------------------------------------------------------------------------ decode families

def _changed(a: bytes, b: bytes, sel=None):
    fa, fb = a.split(b"\t"), b.split(b"\t")
    return [c for c in range(len(fa)) if fa[c] != fb[c] and (sel is None or c in sel)]


INT_T, TXT_T, CHR_T = "int(11)", "varchar(255)", "char(1)"


def _int_change(rng, v, same_len):
    s = b"%d" % v
    if same_len:
        lo, hi = (0, 9) if len(s) == 1 else (10 ** (len(s) - 1), 10 ** len(s) - 1)
        while True:
            n = rng.randint(lo, hi)
            if n != v:
                return n
    if v >= 10 and (v >= 10 ** 8 or rng.random() < 0.5):
        return v // 10  # one digit less
    return v * 10 + rng.randrange(1, 10) if v else rng.randrange(10, 100)  # one digit more


def _txt_change(rng, v, same_len):
    if same_len and v:
        i = rng.randrange(len(v))
        return v[:i] + bytes([rng.choice([c for c in ALPHA if c != v[i]])]) + v[i + 1:]
    n = len(v)
    m = rng.choice([k for k in range(0, 13) if k != n])
    return _txt(rng, m)


def _chr_change(rng, v):
    return bytes([rng.choice([c for c in ALPHA if c != v[0]])])


D1_NCOLS = 300
D1_TAIL = 8                # the last 8 columns hold one byte each: the row's last 16 bytes
D1_SEL = frozenset(range(0, D1_NCOLS, 2))   # the projection of "about half the columns in file order"
D1_M = [0, 1, 31, 32, 33, 63, 64, 65, 66, 128, "all"]


def _d1_types():
    t = [(INT_T, TXT_T, CHR_T)[c % 3] for c in range(D1_NCOLS - D1_TAIL)]
    return t + [CHR_T if c % 2 else INT_T for c in range(D1_TAIL)]


def d1_family():
    """About 300 columns; each row changes exactly m columns against the row before, m cycling through D1_M, the
    changed columns contiguous, spread out or all in the row's last 16 bytes, half of them (where they can) changing
    length.  Then rows with 63, 64 or 65 changes in D1_SEL (or in its complement) and 40 more outside it."""
    rng = random.Random(41)
    types = _d1_types()
    tail = set(range(D1_NCOLS - D1_TAIL, D1_NCOLS))

    def fresh(c):
        t = types[c]
        if c in tail:
            return b"%d" % rng.randrange(10) if t == INT_T else _txt(rng, 1)
        return b"%d" % rng.randrange(10 ** 6) if t == INT_T else _txt(rng, 1) if t == CHR_T else _txt(rng, rng.randrange(13))

    def change(c, v):
        t = types[c]
        same = c in tail or rng.random() < 0.5
        if t == CHR_T:
            return _chr_change(rng, v)
        if t == INT_T:
            return b"%d" % _int_change(rng, int(v), same)
        return _txt_change(rng, v, same)

    cur = [fresh(c) for c in range(D1_NCOLS)]
    rows, claims = [b"\t".join(cur)], []

    def step(cols):
        for c in cols:
            cur[c] = change(c, cur[c])
        rows.append(b"\t".join(cur))

    for rep in range(3):
        for m in D1_M:
            for pat in ("contiguous", "spread", "last16"):
                mm = D1_NCOLS if m == "all" else m
                if pat == "contiguous":
                    s = rng.randrange(D1_NCOLS - mm + 1)
                    cols = list(range(s, s + mm))
                elif pat == "spread":
                    cols = rng.sample(range(D1_NCOLS), mm)
                else:
                    mm = min(mm, D1_TAIL)
                    cols = rng.sample(sorted(tail), mm)
                step(cols)
                claims.append(("changes", len(rows) - 1, mm))
    for sel in (D1_SEL, frozenset(range(D1_NCOLS)) - D1_SEL):
        for k in (63, 64, 65, 64, 63, 65):
            cols = rng.sample(sorted(sel), k) + rng.sample(sorted(set(range(D1_NCOLS)) - sel), 40)
            step(cols)
            claims.append(("changes", len(rows) - 1, k + 40))
            claims.append(("selected_changes", len(rows) - 1, k, 0 in sel))
            step(rng.sample(range(D1_NCOLS), 3))  # a quiet row in between
            claims.append(("changes", len(rows) - 1, 3))
    desc = corpus.desc([(f"c{c}", t) for c, t in enumerate(types)])
    return ("D1_change_counts", desc, _join(rows), True, _group(claims))


def d2_family():
    """Clusters of 8-24 adjacent 1-3-byte columns (ints 9/10/100, texts ""/a/ab/abc): in most rows many of them change
    length, with same-length changes in between.  Column 0 is a varchar of 0-31 bytes that changes in every row, so the
    clusters land at every offset mod 16; the last column changes too."""
    rng = random.Random(42)
    ints = {1: [b"7", b"9", b"3"], 2: [b"10", b"42", b"99"], 3: [b"100", b"512", b"999"]}
    txts = {0: [b""], 1: [b"a", b"b", b"z"], 2: [b"ab", b"cd", b"zz"], 3: [b"abc", b"xyz"]}
    cols, kinds = [("lead", TXT_T)], ["lead"]
    for k in range(6):
        for j in range(rng.randint(8, 24)):
            kind = "int" if k % 2 == 0 else "txt"
            cols.append((f"k{k}_{j}", INT_T if kind == "int" else TXT_T))
            kinds.append(kind)
        cols.append((f"sep{k}", TXT_T))
        kinds.append("sep")
    cols.append(("last", INT_T))
    kinds.append("last")
    pools = {"int": ints, "txt": txts}

    def val(kind, length=None):
        p = pools[kind]
        return rng.choice(p[length if length is not None else rng.choice(sorted(p))])

    cur = []
    for c, kind in enumerate(kinds):
        cur.append(b"" if kind == "lead" else _txt(rng, 5 + c % 15) if kind == "sep" else b"0" if kind == "last"
                   else val(kind))
    rows, claims = [], []
    for r in range(320):
        cur[0] = _txt(rng, (r * 7) % 32)
        moved = 1 if r and len(cur[0]) != (((r - 1) * 7) % 32) else 0
        for c, kind in enumerate(kinds):
            if kind in ("int", "txt") and rng.random() < 0.5:
                old = cur[c]
                if rng.random() < 0.6:
                    cur[c] = val(kind, rng.choice([n for n in pools[kind] if n != len(old)]))
                    moved += 1
                else:
                    alts = [v for v in pools[kind][len(old)] if v != old]
                    if alts:
                        cur[c] = rng.choice(alts)
        if r % 4 != 3:
            old = cur[-1]
            cur[-1] = b"%d" % ((r * 37) % 1000)
            moved += len(old) != len(cur[-1])
        rows.append(b"\t".join(cur))
        if r:
            claims.append(("moved", r, moved))
    desc = corpus.desc(cols)
    return ("D2_moved_clusters", desc, _join(rows), True, _group(claims))


D3_BLOCKS = [1, 2, 31, 32, 33, 65, 100_000]
D3_DESC = corpus.desc([("n", INT_T), ("s", "varchar(64)"), ("c", CHR_T)])


def d3_families():
    """Rows of 5-40 bytes (shorter than a 16-byte chunk, some of them) in blocks of 1 .. 100 000 rows."""
    out = []
    for nrows in D3_BLOCKS:
        rng = random.Random(4300 + nrows)
        cur = [b"1", b"", b"a"]
        rows = []
        for _ in range(nrows):
            if rng.random() < 0.5:
                cur[0] = b"%d" % rng.choice([rng.randrange(10), rng.randrange(100000)])
            if rng.random() < 0.5:
                cur[1] = _txt(rng, rng.choice([0, 0, 1, 2, 5, 15, 16, 17, 30]))
            if rng.random() < 0.3:
                cur[2] = _txt(rng, 1)
            rows.append(b"\t".join(cur))
        out.append((f"D3_short_rows_{nrows}", D3_DESC, _join(rows), True, {"rows": [(0, nrows)]}))
    return out


D4_LENGTHS = [15, 16, 17, 31, 32, 33, 127, 128, 129, 1000, 5000]
D4_DESC = corpus.desc([("a", INT_T), ("t", "text"), ("b", TXT_T), ("t2", "text"), ("c", INT_T)])


def d4_family():
    """Long texts that change by one byte at the start, the middle or the end (same length) or grow or shrink by one
    byte, next to short items that change length."""
    rng = random.Random(44)
    rows, claims = [], []
    shorts = [b"9", b"10", b"100", b"7"]
    sb = [b"", b"a", b"ab", b"x"]
    for L in D4_LENGTHS:
        base = _txt(rng, L)
        other = _txt(rng, 40)
        s1 = _poke(base, 0, lambda b: b ^ 1)
        s2 = _poke(s1, L // 2, lambda b: b ^ 1)
        s3 = _poke(s2, L - 1, lambda b: b ^ 1)
        seq = [("base", base), ("start", s1), ("middle", s2), ("end", s3), ("grow", s3 + b"q"), ("shrink", s3),
               ("shrink", s3[:-1]), ("grow", s3), ("base", s3)]
        for i, (kind, t) in enumerate(seq):
            rows.append(b"\t".join([shorts[i % 4], t, sb[(i + 1) % 4], other if i % 2 else t, b"%d" % (i * 11)]))
            if i:
                claims.append(("long_change", len(rows) - 1, 1, L, kind))
    return ("D4_long_values", D4_DESC, _join(rows), True, _group(claims))


@lru_cache(maxsize=None)
def decode_families():
    return [d1_family(), d2_family()] + d3_families() + [d4_family()]


PROJECTED = ("D1_change_counts", "D2_moved_clusters", "D4_long_values")
