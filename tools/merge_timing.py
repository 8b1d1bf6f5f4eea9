#!/usr/bin/env python
"""merge_timing.py -- kernel times of zdwb_merge_codes against the decode that produced its codes and the host route.

  python tools/merge_timing.py [--c4-blocks 16] [--c4-rows 131072] [--c5-blocks 4] [--c5-rows 262144] [--rounds 5]
                               [--host-columns 3] [--out FILE]

Two workloads, one on each side of the cost:
  c4   bench.Synth blocks, encoded by the library; every used text-like column merged over all blocks.  Low to medium
       cardinality: most strings are shared between blocks.
  c5   tests/c5_check.make_rows blocks: columns k and v hold a distinct 65-byte string per row, w 97 values.
Every round first decodes every block's text-like columns (zdwb_decode_columns, kernel time summed over the blocks),
then merges every column once (kernel time per column, and per kernel summed over the columns); the medians over rounds
are reported.  After those rounds every column's merge is timed again on the wall clock (the whole call: host round
trips and the copies of the outputs included; timing events off), median of --rounds calls.  Per column: input
references (distinct codes per block, summed), distinct output entries, and the bytes the merge reads and writes at the
least (codes in and out, the referenced strings and the output dictionary).  The host route - copy the block
dictionaries and codes to the host, sorted(set()) of the referenced strings, a numpy remap - is timed on the
--host-columns columns with the most references, and one column's result is checked against it.  Prints a summary and
one JSON line (also written to --out) with the card's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from columns_util import TEXT_LIKE  # noqa: E402


def _c4_blocks(ctx, torch, nblocks, rows):
    import bench
    synth = bench.Synth()
    types = synth.schema.types
    cap = synth.cap_for(rows)
    buf = (C.c_uint8 * cap)()
    out = []
    for b in range(nblocks):
        n = synth.block_into(b, rows, C.addressof(buf), cap)
        out.append(ctx.encode_block(types, bytes((C.c_uint8 * n).from_address(C.addressof(buf)))).data)
    return types, out


def _c5_blocks(ctx, torch, nblocks, rows):
    import c5_check
    import oracle as O
    types = O.parse_desc(c5_check.DESC).types
    tsv = c5_check.make_rows(nblocks * rows)
    out, pos = [], 0
    while pos < len(tsv):
        enc = ctx.encode_block(types, tsv[pos:], max_rows=rows)
        out.append(enc.data)
        pos += enc.tsv_consumed
    return types, out


def _host_route(torch, blocks, k):
    """Today's route without a merge kernel: everything to the host, sorted(set()), a numpy remap."""
    import numpy as np
    t0 = time.perf_counter()
    per = []
    for b in blocks:
        d = b.dict.cpu().numpy().tobytes()
        eo = b.entry_off.cpu().numpy()
        codes = b.values[k].cpu().numpy()
        used = np.unique(codes[codes >= 0])
        per.append((codes, used, [d[eo[u]:eo[u + 1] - 1] for u in used.tolist()]))
    ents = sorted(set(s for _, _, strs in per for s in strs))
    where = {s: i for i, s in enumerate(ents)}
    out = []
    for codes, used, strs in per:
        lut = np.full(int(used[-1]) + 2 if used.size else 1, -1, dtype=np.int64)
        lut[used] = [where[s] for s in strs]
        out.append(np.where(codes >= 0, lut[codes], -1))
    res = np.concatenate(out)
    return time.perf_counter() - t0, ents, res


def _workload(ctx, torch, name, types, zs, rounds, host_columns):
    text = [c for c in range(len(types)) if types[c] in TEXT_LIKE]
    probe = [ctx.decode_columns(types, z, text) for z in zs]
    used = [k for k in range(len(text)) if int(torch.stack([b.values[k].max() for b in probe]).max()) >= 0]
    cols = [text[k] for k in used]
    del probe
    ctx.set_tuning("kernel_timing", 1)
    dec_ms, merge_ms, merge_kernels = [], {c: [] for c in cols}, {}
    blocks = None
    for rnd in range(rounds + 1):  # round 0 warms up
        blocks = None
        ctx.kernel_times()
        blocks = [ctx.decode_columns(types, z, cols) for z in zs]
        kt = ctx.kernel_times()
        if rnd:
            dec_ms.append(sum(ms for _, ms in kt.values()))
        per_kernel = {}
        for k, c in enumerate(cols):
            ctx.merge_codes([(b.dict, b.entry_off, b.values[k]) for b in blocks])
            kt = ctx.kernel_times()
            if rnd:
                merge_ms[c].append(sum(ms for _, ms in kt.values()))
                for kn, (_, ms) in kt.items():
                    per_kernel[kn] = per_kernel.get(kn, 0.0) + ms
        for kn, ms in per_kernel.items():
            merge_kernels.setdefault(kn, []).append(ms)
    ctx.set_tuning("kernel_timing", 0)
    # wall time of the whole call, host round trips and the copies of the outputs included, without the timing events
    wall_ms = {c: [] for c in cols}
    for _ in range(rounds):
        for k, c in enumerate(cols):
            parts = [(b.dict, b.entry_off, b.values[k]) for b in blocks]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.merge_codes(parts)
            torch.cuda.synchronize()
            wall_ms[c].append((time.perf_counter() - t0) * 1000)

    per_col = []
    for k, c in enumerate(cols):
        m = ctx.merge_codes([(b.dict, b.entry_off, b.values[k]) for b in blocks])
        refs = sum(int(torch.unique(b.values[k][b.values[k] >= 0]).numel()) for b in blocks)
        n = int(m.codes.numel())
        ref_bytes = 0
        for b in blocks:
            u = torch.unique(b.values[k][b.values[k] >= 0])
            ref_bytes += int((b.entry_off[u + 1] - b.entry_off[u]).sum()) if u.numel() else 0
        moved = 16 * n + ref_bytes + int(m.dict.numel()) + 8 * (m.entries + 1)
        per_col.append({"column": c, "refs": refs, "entries": m.entries, "codes": n, "bytes_moved": moved,
                        "merge_ms": round(statistics.median(merge_ms[c]), 4),
                        "merge_wall_ms": round(statistics.median(wall_ms[c]), 4)})
    per_col.sort(key=lambda x: -x["refs"])

    host = []
    for i, pc in enumerate(per_col[:host_columns]):
        k = cols.index(pc["column"])
        secs, ents, res = _host_route(torch, blocks, k)
        pc["host_route_ms"] = round(secs * 1000, 2)
        host.append(pc["column"])
        if i == 0:  # the GPU result equals the host route's
            m = ctx.merge_codes([(b.dict, b.entry_off, b.values[k]) for b in blocks])
            assert m.strings() == [None if v < 0 else ents[v] for v in res.tolist()], f"{name}: merge differs from the host route"
            assert m.codes.cpu().numpy().tolist() == res.tolist()
    total_merge = sum(x["merge_ms"] for x in per_col)
    return {"workload": name, "blocks": len(zs), "rows": sum(b.nrows for b in blocks), "text_columns": len(cols),
            "decode_columns_ms_all_blocks": round(statistics.median(dec_ms), 4),
            "merge_ms_all_columns": round(total_merge, 4),
            "merge_wall_ms_all_columns": round(sum(x["merge_wall_ms"] for x in per_col), 4),
            "merge_kernels_ms_all_columns": dict(sorted(((kn, round(statistics.median(x), 4)) for kn, x in merge_kernels.items()),
                                                        key=lambda kv: -kv[1])),
            "merge_ms_per_column_median": round(statistics.median(x["merge_ms"] for x in per_col), 4),
            "refs_total": sum(x["refs"] for x in per_col), "entries_total": sum(x["entries"] for x in per_col),
            "checked_column": host[0] if host else None, "columns": per_col}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c4-blocks", type=int, default=16)
    ap.add_argument("--c4-rows", type=int, default=131072)
    ap.add_argument("--c5-blocks", type=int, default=4)
    ap.add_argument("--c5-rows", type=int, default=262144)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--host-columns", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from zdw_b200 import Context

    ctx = Context(0)
    result = {"rounds": args.rounds, "workloads": []}
    for name, make, nb, rows in (("c4", _c4_blocks, args.c4_blocks, args.c4_rows), ("c5", _c5_blocks, args.c5_blocks, args.c5_rows)):
        types, zs = make(ctx, torch, nb, rows)
        w = _workload(ctx, torch, name, types, zs, args.rounds, args.host_columns)
        result["workloads"].append(w)
        top = w["columns"][:3]
        print(f"{name}: {w['blocks']} blocks, {w['rows']} rows, {w['text_columns']} text columns; decode_columns "
              f"{w['decode_columns_ms_all_blocks']:.3f} ms, merges {w['merge_ms_all_columns']:.3f} ms in all; largest: "
              + "; ".join(f"col {x['column']}: {x['refs']} refs -> {x['entries']} entries, {x['merge_ms']:.3f} ms "
                          f"(wall {x['merge_wall_ms']:.3f} ms)"
                          + (f" (host route {x['host_route_ms']:.0f} ms)" if "host_route_ms" in x else "") for x in top),
              flush=True)
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
