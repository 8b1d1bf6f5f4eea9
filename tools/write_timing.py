#!/usr/bin/env python
"""write_timing.py -- what writing a block from typed columns costs: zdwb_render_columns against the encode and the
decode around it.

  python tools/write_timing.py [--blocks 4] [--rows 131072] [--rounds 5] [--out FILE]

bench.Synth (C4-shaped) blocks of --rows rows are encoded by the library and decoded into typed columns (every column,
zdwb_decode_columns).  Each round then runs, per block and in this order: render_columns of the block's columns,
encode_block of the rendered text (input on the device), decode_columns of the block, and write_table of the block as a
one-block raw file under a temporary directory.  Kernel times come from CUDA events (kernel_timing on; every kernel of
the call summed), write_table is timed on the wall clock; each figure is the median over rounds of the per-block mean.
Rendered GB/s = rendered bytes / render kernel time.  Prints a summary and one JSON line (also written to --out) with the
card's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def _kernel_ms(ctx, prefix=None):
    return sum(ms for name, (_, ms) in ctx.kernel_times().items() if prefix is None or name.startswith(prefix))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--rows", type=int, default=131072)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import bench
    from columns_util import TEXT_LIKE
    from zdw_b200 import ColumnTable, Context, FileHeader, write_table

    synth = bench.Synth()
    types = synth.schema.types
    nc = len(types)
    hdr = FileHeader(11, {}, [f"c{k}" for k in range(nc)], list(types), [0] * nc, 0)
    cap = synth.cap_for(args.rows)
    buf = (C.c_uint8 * cap)()
    ctx = Context(0)
    blocks = []
    for b in range(args.blocks):
        n = synth.block_into(b, args.rows, C.addressof(buf), cap)
        z = ctx.encode_block(types, bytes((C.c_uint8 * n).from_address(C.addressof(buf)))).data
        cb = ctx.decode_columns(types, z, list(range(nc)))
        dicts = [(cb.dict, cb.entry_off) if t in TEXT_LIKE else None for t in types]
        blocks.append((z, cb, dicts, n))
    ctx.set_tuning("kernel_timing", 1)
    rows = {k: [] for k in ("render_ms", "render_lengths_ms", "render_write_ms", "render_entries_ms", "encode_ms",
                            "decode_columns_ms", "write_table_ms")}
    rendered = []
    with tempfile.TemporaryDirectory(prefix="zdw_write_timing_") as tmp:
        out_path = Path(tmp) / "block.zdw"
        for rnd in range(args.rounds + 1):  # round 0 warms up every shape
            acc = {k: 0.0 for k in rows}
            for z, cb, dicts, _ in blocks:
                ctx.kernel_times()
                ptr, length = ctx.render_columns(types, cb.values, dicts)
                kt = ctx.kernel_times()
                acc["render_ms"] += sum(ms for _, ms in kt.values())
                acc["render_lengths_ms"] += kt.get("k_render_lengths", (0, 0.0))[1]
                acc["render_write_ms"] += kt.get("k_render_write", (0, 0.0))[1]
                acc["render_entries_ms"] += kt.get("k_render_entries", (0, 0.0))[1]
                if rnd == 0:
                    rendered.append(length)
                ctx.encode_block(types, ptr, length, input_on_device=True)
                acc["encode_ms"] += _kernel_ms(ctx)
                ctx.decode_columns(types, z, list(range(nc)))
                acc["decode_columns_ms"] += _kernel_ms(ctx)
                table = ColumnTable(cb.values, dicts, list(range(nc)), [cb.nrows])
                t0 = time.perf_counter()
                write_table(out_path, hdr, table)
                acc["write_table_ms"] += (time.perf_counter() - t0) * 1e3
            if rnd:
                for k in rows:
                    rows[k].append(acc[k] / len(blocks))
    med = {k: statistics.median(v) for k, v in rows.items()}
    mean_bytes = sum(rendered) / len(rendered)
    result = {"blocks": args.blocks, "rows_per_block": args.rows, "columns": nc, "rounds": args.rounds,
              "rendered_bytes_per_block": mean_bytes, "synth_tsv_bytes_per_block": sum(b[3] for b in blocks) / len(blocks),
              "per_block": {k: round(v, 4) for k, v in med.items()},
              "render_gb_s": round(mean_bytes / (med["render_ms"] * 1e-3) / 1e9, 2),
              "render_write_gb_s": round(mean_bytes / (med["render_write_ms"] * 1e-3) / 1e9, 2)}
    result["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                   capture_output=True, text=True).stdout.strip()
    print(f"C4 blocks of {args.rows} rows, {mean_bytes / 1e6:.1f} MB rendered per block: render {med['render_ms']:.3f} ms "
          f"({result['render_gb_s']} GB/s; lengths {med['render_lengths_ms']:.3f}, write {med['render_write_ms']:.3f}, "
          f"entries {med['render_entries_ms']:.3f}), encode {med['encode_ms']:.3f} ms, decode_columns "
          f"{med['decode_columns_ms']:.3f} ms, write_table wall {med['write_table_ms']:.1f} ms", flush=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
