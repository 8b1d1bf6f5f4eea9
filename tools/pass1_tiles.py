#!/usr/bin/env python
"""pass1_tiles.py -- per-kernel encode times of C4 blocks for several values of one tuning knob, alternated.

  python tools/pass1_tiles.py --knob enc_dtile=32768,65536,131072 [--blocks 4] [--rounds 5] [--out FILE]

Every round encodes each block once per knob value (values in turn, so that drift of the clock or of other work on the
GPU spreads over all of them) with the instrumented kernel times (`kernel_timing`), and checks that the encoded bytes do
not depend on the knob.  Prints, per value, the median over rounds of every kernel's ms per block, and the same as one
JSON line (also written to --out).
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--knob", required=True, help="name=v1,v2,...")
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--rows", type=int, default=131072)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import bench
    from zdw_b200 import Context

    name, vals = args.knob.split("=")
    values = [int(x) for x in vals.split(",")]
    synth = bench.Synth()
    types = synth.schema.types
    dev = torch.device("cuda", 0)
    cap = synth.cap_for(args.rows)
    buf = (C.c_uint8 * cap)()
    blocks = []
    for b in range(args.blocks):
        n = synth.block_into(b, args.rows, C.addressof(buf), cap)
        t = torch.empty(n + 64, dtype=torch.uint8, device=dev)
        t[:n].copy_(torch.frombuffer((C.c_uint8 * n).from_address(C.addressof(buf)), dtype=torch.uint8))
        blocks.append((t, n))
    torch.cuda.synchronize()
    ctx = Context(0)
    ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    ctx.set_tuning("kernel_timing", 1)

    ref = {}
    times = {v: {} for v in values}  # value -> kernel -> [ms per block, one per round]
    for rnd in range(args.rounds + 1):  # round 0 warms every value up and records the bytes
        for v in values:
            ctx.set_tuning(name, v)
            ctx.kernel_times()
            for j, (t, n) in enumerate(blocks):
                blk = ctx.encode_block(types, t.data_ptr(), n, input_on_device=True, output_on_device=True)
                z = torch.empty(blk.length, dtype=torch.uint8, device=dev)
                bench._d2d(torch, z, blk.dev_ptr, blk.length)
                if j not in ref:
                    ref[j] = z
                else:
                    assert ref[j].numel() == blk.length and bool((ref[j] == z).all()), f"block {j}: bytes differ at {name}={v}"
            kt = ctx.kernel_times()
            if rnd:
                for k, (cnt, ms) in kt.items():
                    times[v].setdefault(k, []).append(ms / len(blocks))

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    result = {"knob": name, "blocks": args.blocks, "rows_per_block": args.rows, "rounds": args.rounds, "gpu": gpu,
              "ms_per_block": {}}
    for v in values:
        med = {k: round(statistics.median(x), 4) for k, x in times[v].items()}
        med = dict(sorted(med.items(), key=lambda kv: -kv[1]))
        total = round(sum(med.values()), 4)
        result["ms_per_block"][str(v)] = {"total": total, **med}
        top = list(med.items())[:5]
        print(f"{name}={v}: total={total:.3f} " + " ".join(f"{k}={ms:.3f}" for k, ms in top), flush=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
