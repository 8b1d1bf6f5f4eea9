#!/usr/bin/env python
"""match_timing.py -- kernel and wall times of zdwb_match_like and zdwb_find_strings against the host route.

  python tools/match_timing.py [--c5-blocks 4] [--c5-rows 262144] [--c4-blocks 4] [--c4-rows 131072] [--urls 200000]
                               [--rounds 5] [--out FILE]

Workloads:
  c5        column k of tests/c5_check.make_rows blocks merged over all blocks (about 1 M distinct 65-byte strings):
            LIKE 'abc%', '%abc%', '%a_c%d', and '%ABC%' with ignore_case; 1 M lookups, half of them present.
  c4        every used text-like column of bench.Synth blocks merged over all blocks (what read_table does): LIKE '%a%'
            and 1000 lookups per column.
  urls      URL-like entries of 200 to 4096 bytes ('%/checkout%', '%abc%'), and the same number of entries all of the
            mean length ("urls_uniform"): equal bytes, no spread of lengths within a warp.
Kernel times come from CUDA events (kernel_timing), medians of --rounds rounds; L2 is overwritten (a 512 MB memset on
torch's stream) before every timed call.  The wall time is that of the whole Context call (host round trip and the copy
of the outputs included, timing events off) on a warm context, and with a context created for the call, as the
predicates module does.  "bytes" is what a call must read and write at the least: the offsets and bytes of every entry
and the flags for LIKE; that plus the query bytes and offsets and the ranks and found flags for the lookups.  The host
route copies the dictionary out, builds one bytes per entry, and runs re.fullmatch (LIKE) or bisect (lookup) per
entry / query; its answers are checked against the GPU's.  Prints one JSON line (also written to --out) with the card's
name, power limit and max SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import bisect
import json
import random
import re
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))

from columns_util import TEXT_LIKE  # noqa: E402


def like_regex(pattern: bytes, ignore_case: bool):
    """The LIKE pattern (escape '\\') as a compiled bytes regex for re.fullmatch."""
    out, i = [], 0
    while i < len(pattern):
        c = pattern[i:i + 1]
        if c == b"\\":
            i += 1
            out.append(re.escape(pattern[i:i + 1]))
        elif c == b"%":
            out.append(b".*")
        elif c == b"_":
            out.append(b".")
        else:
            out.append(re.escape(c))
        i += 1
    return re.compile(b"".join(out), re.S | (re.I if ignore_case else 0))


def host_entries(dct, eo):
    d = dct.cpu().numpy().tobytes()
    offs = eo.cpu().tolist()
    return [d[a:b - 1] for a, b in zip(offs, offs[1:])]


class Timer:
    def __init__(self, ctx, torch, rounds):
        self.ctx, self.torch, self.rounds = ctx, torch, rounds
        self.flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def kernels(self, call):
        """(median kernel ms, {kernel: median ms}) of call() over the rounds, L2 overwritten before each"""
        ctx, torch = self.ctx, self.torch
        call()  # warm-up
        ctx.set_tuning("kernel_timing", 1)
        tot, per = [], {}
        for _ in range(self.rounds):
            self.flush.zero_()
            torch.cuda.synchronize()
            ctx.kernel_times()
            call()
            kt = ctx.kernel_times()
            tot.append(sum(ms for _, ms in kt.values()))
            for k, (_, ms) in kt.items():
                per.setdefault(k, []).append(ms)
        ctx.set_tuning("kernel_timing", 0)
        return statistics.median(tot), {k: round(statistics.median(v), 4) for k, v in per.items()}

    def wall(self, call):
        torch = self.torch
        ms = []
        for _ in range(self.rounds):
            self.flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            call()
            torch.cuda.synchronize()
            ms.append((time.perf_counter() - t0) * 1000)
        return statistics.median(ms)


def like_case(tm, Context, dct, eo, pattern, ic, ents, host=True):
    ctx = tm.ctx
    E = eo.numel() - 1
    k_ms, per = tm.kernels(lambda: ctx.match_like(dct, eo, pattern, ignore_case=ic))
    w_ms = tm.wall(lambda: ctx.match_like(dct, eo, pattern, ignore_case=ic))

    def fresh():
        with Context(0) as c:
            c.match_like(dct, eo, pattern, ignore_case=ic)
    f_ms = tm.wall(fresh)
    nbytes = int(dct.numel()) + 8 * (E + 1) + (E + 1)
    r = {"pattern": pattern.decode("latin1"), "ignore_case": ic, "entries": E, "bytes": nbytes, "kernel_ms": round(k_ms, 4),
         "gb_per_s": round(nbytes / k_ms / 1e6, 1), "kernels": per, "wall_ms": round(w_ms, 4),
         "wall_fresh_context_ms": round(f_ms, 3)}
    if host:
        t0 = time.perf_counter()
        he = host_entries(dct, eo)
        rx = like_regex(pattern, ic)
        want = [rx.fullmatch(s) is not None for s in he]
        r["host_route_ms"] = round((time.perf_counter() - t0) * 1000, 2)
        got = ctx.match_like(dct, eo, pattern, ignore_case=ic)[:-1].cpu().tolist()
        assert got == want, f"match_like differs from the host route for {pattern!r}"
        r["matches"] = sum(want)
    return r


def find_case(tm, Context, dct, eo, queries, host=True):
    ctx = tm.ctx
    E = eo.numel() - 1
    k_ms, per = tm.kernels(lambda: ctx.find_strings(dct, eo, queries))
    w_ms = tm.wall(lambda: ctx.find_strings(dct, eo, queries))
    qb = sum(len(q) for q in queries)
    nbytes = int(dct.numel()) + 8 * (E + 1) + qb + 8 * (len(queries) + 1) + 9 * len(queries)
    r = {"queries": len(queries), "entries": E, "bytes": nbytes, "kernel_ms": round(k_ms, 4),
         "gb_per_s": round(nbytes / k_ms / 1e6, 1), "kernels": per, "wall_ms": round(w_ms, 4)}
    if host:
        t0 = time.perf_counter()
        he = host_entries(dct, eo)
        want = [bisect.bisect_left(he, q) for q in queries]
        r["host_route_ms"] = round((time.perf_counter() - t0) * 1000, 2)
        rank, found = ctx.find_strings(dct, eo, queries)
        assert rank.cpu().tolist() == want, "find_strings differs from bisect"
        r["found"] = int(found.sum())
    return r


def dev_dict(torch, ents):
    import numpy as np
    lens = np.fromiter((len(e) + 1 for e in ents), dtype=np.int64, count=len(ents))
    eo = np.empty(len(ents) + 1, dtype=np.int64)
    eo[0] = 1
    np.cumsum(lens, out=eo[1:])
    eo[1:] += 1
    d = b"\0" + b"".join(e + b"\0" for e in ents)
    return torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda(), torch.from_numpy(eo).cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c5-blocks", type=int, default=4)
    ap.add_argument("--c5-rows", type=int, default=262144)
    ap.add_argument("--c4-blocks", type=int, default=4)
    ap.add_argument("--c4-rows", type=int, default=131072)
    ap.add_argument("--urls", type=int, default=200000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import merge_timing
    from zdw_b200 import Context

    ctx = Context(0)
    tm = Timer(ctx, torch, args.rounds)
    result = {"rounds": args.rounds}
    rng = random.Random(1)

    # ---- c5: one merged column of about 1 M distinct 65-byte strings
    types, zs = merge_timing._c5_blocks(ctx, torch, args.c5_blocks, args.c5_rows)
    k = next(c for c in range(len(types)) if types[c] in TEXT_LIKE)
    blocks = [ctx.decode_columns(types, z, [k]) for z in zs]
    m = ctx.merge_codes([(b.dict, b.entry_off, b.values[0]) for b in blocks])
    del blocks
    dct, eo = m.dict, m.entry_off
    ents = host_entries(dct, eo)
    c5 = {"entries": len(ents), "dict_bytes": int(dct.numel()), "like": [], "find": None}
    for p, ic in ((b"abc%", False), (b"%abc%", False), (b"%a_c%d", False), (b"%ABC%", True)):
        c5["like"].append(like_case(tm, Context, dct, eo, p, ic, ents))
        print("c5 like", c5["like"][-1], flush=True)
    qs = [ents[rng.randrange(len(ents))] if rng.random() < 0.5 else ents[rng.randrange(len(ents))][:-1] + b"~"
          for _ in range(1 << 20)]
    c5["find"] = find_case(tm, Context, dct, eo, qs)
    print("c5 find", c5["find"], flush=True)
    result["c5"] = c5
    del m, dct, eo, ents

    # ---- c4: every used text column of a multi-block table
    types, zs = merge_timing._c4_blocks(ctx, torch, args.c4_blocks, args.c4_rows)
    text = [c for c in range(len(types)) if types[c] in TEXT_LIKE]
    blocks = [ctx.decode_columns(types, z, text) for z in zs]
    cols = []
    for j, c in enumerate(text):
        if int(torch.stack([b.values[j].max() for b in blocks]).max()) < 0:
            continue
        mm = ctx.merge_codes([(b.dict, b.entry_off, b.values[j]) for b in blocks])
        cols.append((c, mm.dict, mm.entry_off))
    del blocks
    rows_like, rows_find = [], []
    big = sorted(cols, key=lambda x: -x[2].numel())[:3]
    for c, d, e in cols:
        he = host_entries(d, e)
        q = [he[rng.randrange(len(he))] for _ in range(1000)]
        host = any(c == b[0] for b in big)
        rl = like_case(tm, Context, d, e, b"%a%", False, he, host)
        rf = find_case(tm, Context, d, e, q, host)
        rl["column"] = rf["column"] = c
        rows_like.append(rl)
        rows_find.append(rf)
    result["c4"] = {
        "blocks": args.c4_blocks, "rows_per_block": args.c4_rows, "text_columns": len(cols),
        "entries_total": sum(r["entries"] for r in rows_like),
        "like_kernel_ms_all_columns": round(sum(r["kernel_ms"] for r in rows_like), 4),
        "like_kernel_ms_per_column_median": round(statistics.median(r["kernel_ms"] for r in rows_like), 4),
        "like_wall_ms_per_column_median": round(statistics.median(r["wall_ms"] for r in rows_like), 4),
        "like_wall_fresh_context_ms_median": round(statistics.median(r["wall_fresh_context_ms"] for r in rows_like), 3),
        "find_kernel_ms_all_columns": round(sum(r["kernel_ms"] for r in rows_find), 4),
        "find_wall_ms_per_column_median": round(statistics.median(r["wall_ms"] for r in rows_find), 4),
        "largest": [r for r in rows_like if "host_route_ms" in r] + [r for r in rows_find if "host_route_ms" in r]}
    print("c4", {k: v for k, v in result["c4"].items() if k != "largest"}, flush=True)
    del cols

    # ---- long entries: URL-like, 200 B to 4 KiB, against the same number of entries all of the mean length
    alpha = "abcdefghijklmnopqrstuvwxyz0123456789/-_.=&?"
    urls = set()
    while len(urls) < args.urls:
        n = rng.randint(200, 4096)
        body = "".join(rng.choice(alpha) for _ in range(40))
        urls.add(("https://www.example.com/" + body + "/" * (n % 7) + "x" * (n - 64 - n % 7)).encode()[:n])
    urls = sorted(urls)
    mean = sum(len(u) for u in urls) // len(urls)
    uniform = sorted({u[:mean].ljust(mean, b"y") for u in urls})
    for name, ents in (("urls", urls), ("urls_uniform", uniform)):
        d, e = dev_dict(torch, ents)
        result[name] = {"entries": len(ents), "dict_bytes": int(d.numel()),
                        "like": [like_case(tm, Context, d, e, p, False, ents) for p in (b"%/checkout%", b"%abc%")]}
        print(name, result[name], flush=True)
        del d, e

    result["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                   capture_output=True, text=True).stdout.strip()
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
