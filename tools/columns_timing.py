#!/usr/bin/env python
"""columns_timing.py -- per-kernel times of C4 blocks decoded to text and to typed columns, alternated.

  python tools/columns_timing.py [--blocks 4] [--rows 131072] [--rounds 5] [--out FILE]

The C4 blocks are made with bench.Synth and encoded on the device.  Every round decodes each block three ways, in turn,
with the instrumented kernel times (`kernel_timing`):
  rows     zdwb_decode_block, TSV left on the device
  all      zdwb_decode_columns of every used column
  sel16    zdwb_decode_columns of 16 used columns, 8 of them text-like
Before the timed rounds one block's columns are checked against its TSV (NUL-separated in-memory layout).  Prints, per
way, the median over rounds of every kernel's ms per block and the output bytes, and the same as one JSON line (also
written to --out) with the card's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from columns_util import TEXT_LIKE, entries, render  # noqa: E402

def _used_columns(z: bytes, nc: int) -> list:
    """Columns with columnSize != 0: numRows u32 | longestLine u32 | isLast u8 | idxSize u8 | dictionary | columnSize[nc]"""
    isz = z[9]
    dsize = int.from_bytes(z[10:10 + isz], "little") if isz else 0
    cs = z[10 + isz + dsize:10 + isz + dsize + nc]
    return [c for c in range(nc) if cs[c]]


def _check(ctx, types, z: bytes):
    """Every column of one block against the block's own NUL-separated TSV."""
    nc = len(types)
    want = ctx.decode_block(types, z, separator=b"\0").tsv
    cb = ctx.decode_columns(types, z, list(range(nc)))
    d = bytes(cb.dict.cpu().numpy().tobytes())
    ents = entries(d, cb.entry_off.cpu().tolist())
    vals = cb.values.cpu().tolist()
    cols = [[render(types[c], v, ents) for v in vals[c]] for c in range(nc)]
    got = b"".join(b"\0".join(row) + b"\0" for row in zip(*cols))
    assert got == want, "decode_columns disagrees with the TSV of the same block"
    return cb.nrows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--rows", type=int, default=131072)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import bench
    from zdw_b200 import Context

    synth = bench.Synth()
    types = synth.schema.types
    dev = torch.device("cuda", 0)
    cap = synth.cap_for(args.rows)
    buf = (C.c_uint8 * cap)()
    ctx = Context(0)
    ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    blocks = []  # (device tensor holding the encoded block, length)
    for b in range(args.blocks):
        n = synth.block_into(b, args.rows, C.addressof(buf), cap)
        t = torch.empty(n + 64, dtype=torch.uint8, device=dev)
        t[:n].copy_(torch.frombuffer((C.c_uint8 * n).from_address(C.addressof(buf)), dtype=torch.uint8))
        enc = ctx.encode_block(types, t.data_ptr(), n, input_on_device=True, output_on_device=True)
        z = torch.empty(enc.length + 64, dtype=torch.uint8, device=dev)
        bench._d2d(torch, z, enc.dev_ptr, enc.length)
        blocks.append((z, enc.length))
    torch.cuda.synchronize()
    z0 = bytes(blocks[0][0][:blocks[0][1]].cpu().numpy().tobytes())
    checked_rows = _check(ctx, types, z0)

    # the used columns of the first block, and 16 of them with 8 text-like
    used = _used_columns(z0, len(types))
    text = [c for c in used if types[c] in TEXT_LIKE][:8]
    other = [c for c in used if types[c] not in TEXT_LIKE][:16 - len(text)]
    sel16 = sorted(text + other)

    ctx.set_tuning("kernel_timing", 1)
    ways = {
        "rows": lambda z, n: ctx.decode_block(types, z.data_ptr(), n, input_on_device=True, output_on_device=True).length,
        "all": lambda z, n: ctx.decode_columns(types, z.data_ptr(), used, n, input_on_device=True).values.numel() * 8,
        "sel16": lambda z, n: ctx.decode_columns(types, z.data_ptr(), sel16, n, input_on_device=True).values.numel() * 8,
    }
    times = {w: {} for w in ways}
    out_bytes = {w: 0 for w in ways}
    for rnd in range(args.rounds + 1):  # round 0 warms every way up
        for w, f in ways.items():
            ctx.kernel_times()
            nbytes = 0
            for z, n in blocks:
                nbytes += f(z, n)
            kt = ctx.kernel_times()
            out_bytes[w] = nbytes // len(blocks)
            if rnd:
                for k, (cnt, ms) in kt.items():
                    times[w].setdefault(k, []).append(ms / len(blocks))

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    result = {"blocks": args.blocks, "rows_per_block": args.rows, "rounds": args.rounds, "gpu": gpu,
              "used_columns": len(used), "sel16_text_columns": len(text), "checked_rows": checked_rows,
              "output_bytes_per_block": out_bytes, "ms_per_block": {}}
    for w in ways:
        med = {k: round(statistics.median(x), 4) for k, x in times[w].items()}
        med = dict(sorted(med.items(), key=lambda kv: -kv[1]))
        total = round(sum(med.values()), 4)
        result["ms_per_block"][w] = {"total": total, **med}
        top = list(med.items())[:6]
        print(f"{w}: total={total:.3f} ms, {out_bytes[w] / 1e6:.1f} MB out; " + " ".join(f"{k}={ms:.3f}" for k, ms in top),
              flush=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
