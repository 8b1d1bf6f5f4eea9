#!/usr/bin/env python
"""numbers_timing.py -- kernel and wall times of zdwb_parse_numbers and zdwb_format_numbers against the host route.

  python tools/numbers_timing.py [--synth 10000000] [--rounds 5] [--out FILE]

Workloads:
  movie_tickets  the golden's date_time dictionary (every distinct DATETIME of the file) and its revenue dictionary,
                 merged by read_table; parse, format of the parsed values, and the wall time of to_datetime /
                 to_decimal(scale=2) over the table's rows.
  synth          --synth distinct DATETIMEs (whole seconds over 1970..2100) and --synth distinct DECIMALs at scale 2
                 (|v| < 10^12), formatted by zdwb_format_numbers and parsed back.
Kernel times come from CUDA events (kernel_timing), medians of --rounds rounds; L2 is overwritten (a 512 MB memset on
torch's stream) before every timed call, as tools/match_timing.py does.  Wall times are those of the whole Context call
(copy of the outputs included) on a warm context; to_datetime / to_decimal open a context per call.  "bytes" is what a
call must read and write at the least: parse the dictionary, its offsets and the values and flags; format the values,
the dictionary, its offsets and the codes.  The host route copies the dictionary out and parses every entry with
datetime.fromisoformat / decimal.Decimal; its answers are checked against the GPU's, and every formatted dictionary is
parsed back to its values.  Prints one JSON line (also written to --out) with the card's name, power limit and max SM
clock read in the same run.
"""
from __future__ import annotations

import argparse
import datetime as dt
import decimal
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))

from match_timing import Timer, host_entries  # noqa: E402

EPOCH = dt.datetime(1970, 1, 1)
US = dt.timedelta(microseconds=1)


def host_parse(dct, eo, kind, scale):
    """(ms, values) of the host route: the dictionary copied out, one datetime / Decimal per entry"""
    t0 = time.perf_counter()
    ents = host_entries(dct, eo)
    if kind == 0:
        vals = [(dt.datetime.fromisoformat(s.decode()) - EPOCH) // US for s in ents]
    else:
        vals = [int(decimal.Decimal(s.decode()).scaleb(scale)) for s in ents]
    return (time.perf_counter() - t0) * 1000, vals


def parse_case(tm, dct, eo, kind, scale, null):
    ctx = tm.ctx
    E = eo.numel() - 1
    tm.torch.cuda.synchronize()  # the context's stream does not wait for torch's
    k_ms, per = tm.kernels(lambda: ctx.parse_numbers(dct, eo, kind, digits=scale, null_text=null))
    w_ms = tm.wall(lambda: ctx.parse_numbers(dct, eo, kind, digits=scale, null_text=null))
    nbytes = int(dct.numel()) + 8 * (E + 1) + 9 * (E + 1)
    h_ms, want = host_parse(dct, eo, kind, scale)
    values, ok = ctx.parse_numbers(dct, eo, kind, digits=scale, null_text=null)
    assert bool(ok[:-1].all()) and values[:-1].cpu().tolist() == want, "parse_numbers differs from the host route"
    return {"entries": E, "dict_bytes": int(dct.numel()), "bytes": nbytes, "kernel_ms": round(k_ms, 4),
            "gb_per_s": round(nbytes / k_ms / 1e6, 1), "kernels": per, "wall_ms": round(w_ms, 4),
            "host_route_ms": round(h_ms, 1)}, values[:-1]


def format_case(tm, values, kind, digits):
    ctx = tm.ctx
    n = values.numel()
    tm.torch.cuda.synchronize()
    k_ms, per = tm.kernels(lambda: ctx.format_numbers(values, kind, digits=digits))
    w_ms = tm.wall(lambda: ctx.format_numbers(values, kind, digits=digits))
    m = ctx.format_numbers(values, kind, digits=digits)
    back, ok = ctx.parse_numbers(m.dict, m.entry_off, kind, digits=digits)
    import torch
    assert bool(ok[:-1].all()) and torch.equal(back[m.codes], values), "format_numbers does not parse back"
    nbytes = 8 * n + int(m.dict.numel()) + 8 * (n + 1) + 8 * n
    sort_ms = sum(ms for k, ms in per.items() if not k.startswith(("k_num_", "k_scan_")))  # the sort's own scans counted apart
    return {"values": n, "dict_bytes": int(m.dict.numel()), "bytes": nbytes, "kernel_ms": round(k_ms, 4),
            "gb_per_s": round(nbytes / k_ms / 1e6, 1), "sort_kernels_ms": round(sort_ms, 4), "kernels": per,
            "wall_ms": round(w_ms, 4)}, m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--synth", type=int, default=10_000_000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import oracle as O
    from zdw_b200 import Context, read_table, to_datetime, to_decimal

    ctx = Context(0)
    tm = Timer(ctx, torch, args.rounds)
    result = {"rounds": args.rounds}

    # ---- movie_tickets: its two number columns as read_table gives them
    hdr, t = read_table(O.golden("movie_tickets.zdw"))
    mt = {"rows": int(t.values.shape[1])}
    for name, k, kind, scale, null in (("date_time", 0, 0, 0, b""), ("revenue", 5, 1, 2, b"0.000000000000")):
        dct, eo = t.dicts[k]
        r, vals = parse_case(tm, dct, eo, kind, scale, null)
        fmt, _ = format_case(tm, torch.unique(vals), kind, scale if kind else 0)
        to = (lambda: to_datetime(hdr, t, k)) if kind == 0 else (lambda: to_decimal(hdr, t, k, scale=scale))
        r["to_wall_ms"] = round(tm.wall(to), 4)
        mt[name] = {"parse": r, "format": fmt}
        print("movie_tickets", name, mt[name], flush=True)
    result["movie_tickets"] = mt
    del t

    # ---- synthetic: distinct DATETIMEs and DECIMALs, formatted on the GPU, then parsed back
    g = torch.Generator(device="cuda").manual_seed(1)
    synth = {}
    for name, kind, digits, lo, hi in (("datetime", 0, 0, 0, 4_102_444_800), ("decimal_s2", 1, 2, -10 ** 12, 10 ** 12)):
        v = torch.unique(torch.randint(lo, hi, (int(args.synth * 1.02),), generator=g, device="cuda", dtype=torch.int64))
        v = v[torch.randperm(v.numel(), generator=g, device="cuda")[:args.synth]].sort().values.contiguous()
        if kind == 0:
            v *= 1_000_000
        fmt, m = format_case(tm, v, kind, digits)
        r, _ = parse_case(tm, m.dict, m.entry_off, kind, digits, b"")
        synth[name] = {"format": fmt, "parse": r}
        print("synth", name, synth[name], flush=True)
        del m, v
    result["synth"] = synth

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
