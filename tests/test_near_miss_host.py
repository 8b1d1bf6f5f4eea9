"""The near-miss generator (tests/near_miss.py) on the CPU: every claim a family makes holds on its text, and every
canonical family survives the C restatement's round trip.  A claim that does not hold would leave the GPU tests in
test_gpu_near_miss.py exercising something other than what they name."""
import pytest

import near_miss as N
import oracle as O

ENC = N.encode_families()
DEC = N.decode_families()
ALL = ENC + DEC


def _rows(tsv):
    return tsv[:-1].split(b"\n") if tsv.endswith(b"\n") else tsv.split(b"\n")


def _fields(tsv):
    return [r.split(b"\t") for r in _rows(tsv)]


def _diff_at(a, b):
    return [i for i in range(len(a)) if a[i] != b[i]]


@pytest.mark.parametrize("fam", ALL, ids=[f[0] for f in ALL])
def test_claims_hold(fam):
    name, desc, tsv, canonical, claims = fam
    sch = O.parse_desc(desc)
    f = _fields(tsv)
    assert all(len(r) == sch.ncols for r in f), "a row with the wrong number of fields"
    assert b"\\" not in tsv and b"\0" not in tsv
    for r, c, L, off in claims.get("one_off", []):
        a, b = f[r - 1][c], f[r][c]
        assert len(a) == len(b) == L and _diff_at(a, b) == [off], (name, r)
    for r, c in claims.get("repeat", []):
        assert f[r][c] == f[r - 1][c] and f[r][c]
    for r, c, nc in claims.get("neighbour", []):
        v = f[r][c]
        assert v and v == f[r - 1][nc] and v != f[r - 1][c] and len(f[r - 1][c]) in (0, len(v)), (name, r, c)
    for r, c in claims.get("last_byte", []):
        a, b = f[r - 1][c], f[r][c]
        assert len(a) == len(b) and a[-1] != b[-1], (name, r)
    for r, c in claims.get("same_spelling_len", []):
        assert f[r][c] != f[r - 1][c] and len(f[r][c]) == len(f[r - 1][c])
    for r, c in claims.get("trimmed_equal", []):
        assert f[r][c] != f[r - 1][c] and f[r][c].rstrip(b" ") == f[r - 1][c].rstrip(b" ")
    for r, c in claims.get("trimmed_differ", []):
        assert f[r][c].rstrip(b" ") != f[r - 1][c].rstrip(b" ")
    for r, m in claims.get("changes", []):
        assert sum(x != y for x, y in zip(f[r], f[r - 1])) == m, (name, r)
    for r, k, even in claims.get("selected_changes", []):
        sel = N.D1_SEL if even else frozenset(range(N.D1_NCOLS)) - N.D1_SEL
        assert sum(f[r][c] != f[r - 1][c] for c in sel) == k
        assert sum(x != y for x, y in zip(f[r], f[r - 1])) >= 65  # more flagged columns than the delta writer lists
    for r, moved in claims.get("moved", []):
        assert sum(len(x) != len(y) for x, y in zip(f[r], f[r - 1])) == moved, (name, r)
        assert f[r][0] != f[r - 1][0]  # the row's head changes in every row
    for r, c, L, kind in claims.get("long_change", []):
        a, b = f[r - 1][c], f[r][c]
        if kind in ("start", "middle", "end"):
            assert len(a) == len(b) == L and _diff_at(a, b) == [{"start": 0, "middle": L // 2, "end": L - 1}[kind]]
        elif kind == "base":
            assert a == b and len(a) == L
        else:
            assert len(b) - len(a) == (1 if kind == "grow" else -1)
    if "/end" in name:
        # the last row's last field differs from the row before in its last byte, and that byte ends the buffer (or
        # stands in front of the final newline)
        a, b = f[-2][-1], f[-1][-1]
        assert len(a) == len(b) and a[-1] != b[-1]
        assert tsv.endswith(b + (b"\n" if name.endswith("_nl") else b""))
    opts = claims.get("opts", {})
    if opts.get("rows_per_block"):
        rpb = opts["rows_per_block"]
        assert any(r % rpb == 0 for r, *_ in claims["one_off"]), "no block opens with a one-off row"
    if name.startswith("E") and "/small" in name:
        assert len(tsv) < 65536
    if name.startswith("E") and "/mid" in name:
        assert len(tsv) > 256 * 1024


@pytest.mark.parametrize("fam", [f for f in ENC if f[0].startswith("E2") and f[0].endswith("/mid")],
                         ids=[f[0] for f in ENC if f[0].startswith("E2") and f[0].endswith("/mid")])
def test_e2_shape(fam):
    """Rows fit the row-delta pass 1 (at most 280 non-empty fields, under 64 KiB), one row has exactly 280, and the
    neighbour-equal claims cover both directions at every focus pair: across words, across a 1024-column rank round,
    and at column 4095."""
    name, desc, tsv, canonical, claims = fam
    for r in _fields(tsv):
        assert sum(1 for x in r if x) <= N.DCAP
    assert all(len(r) < 65536 for r in _rows(tsv))
    pairs = {(c, nc) for _, c, nc in claims["neighbour"]}
    for a, b in N.E2_FOCUS:
        assert (a, b) in pairs and (b, a) in pairs, (name, a, b)
    if name.startswith("E2_L1/"):
        assert max(sum(1 for x in r if x) for r in _fields(tsv)) == N.DCAP


@pytest.mark.parametrize("L", N.E1_LENGTHS)
def test_e1_alignments(L):
    """The changed field and its copy in the row before sit at every pair of word offsets, and at every distance mod 16."""
    fam = next(f for f in ENC if f[0] == f"E1_L{L}/mid")
    rows = _rows(fam[2])
    starts, pos = [], 0
    for r in rows:
        starts.append(pos + r.rindex(b"\t") + 1)
        pos += len(r) + 1
    words = {(starts[r] % 4, starts[r - 1] % 4) for r, *_ in fam[4]["one_off"]}
    rel = {(starts[r] - starts[r - 1]) % 16 for r, *_ in fam[4]["one_off"]}
    assert len(words) == 16 and rel == set(range(16))


def test_d1_counts_cover_the_list_limit():
    """D1's rows change 0 .. all columns, among them 63, 64, 65 and 66 (the delta writer lists up to 64)."""
    claims = next(f for f in DEC if f[0] == "D1_change_counts")[4]
    ms = {m for _, m in claims["changes"]}
    assert {0, 1, 31, 32, 33, 63, 64, 65, 66, 128, N.D1_NCOLS} <= ms
    assert {k for _, k, _ in claims["selected_changes"]} == {63, 64, 65}


def test_d3_row_lengths():
    for name, desc, tsv, canonical, claims in DEC:
        if name.startswith("D3_"):
            rows = _rows(tsv)
            assert len(rows) == claims["rows"][0][1]
            assert all(2 <= len(r) + 1 <= 40 for r in rows)


@pytest.mark.parametrize("fam", ALL, ids=[f[0] for f in ALL])
def test_oracle_round_trip(fam):
    name, desc, tsv, canonical, claims = fam
    opts = claims.get("opts", {})
    r = O.encode(O.parse_desc(desc), tsv, trim=bool(opts.get("trim")), rows_per_block=opts.get("rows_per_block", 0))
    assert r.rc == 0
    if canonical:
        d = O.decode(r.data)
        assert d.rc == 0
        assert d.tsv == N.expected_tsv(tsv)
