#!/usr/bin/env python
"""bench.py -- TSV->ZDW encode / ZDW->TSV decode throughput of the B200 hot path (BASELINE config C4).

  python bench.py --gpus N --steps K --warmup W              # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle/_ref)

Workload (config C4, SURVEY 8(d)): synthetic analytics-hits-shaped TSV, 2 086 columns (256 populated),
64 blocks of 131 072 rows (about 32 GB) generated from the reference's own analytics-hits fixture with
seed 20190901.  ZDW blocks are independent, so the file is sharded by whole blocks over the N ranks
(strong scaling: the total work is the same at every N) and there is no data-path collective; the host
concatenates blocks in order.  A "step" encodes every block of the rank's shard and decodes it again.

`value`   = encode GB/s, TSV bytes / device time, inputs resident in HBM, outputs left in HBM.
`decode`  = the same for the decoder (ZDW blocks resident in HBM, TSV left in HBM).
`e2e`     = the same metric through the C ABI with HOST buffers: pinned TSV in, host ZDW out (copies timed).
`roofline`= dominant kernel, algorithmic bytes (TSV + ZDW of a block, SURVEY 8(d)) / its mean launch time,
            measured with CUDA events in one instrumented step after the timed steps.
"""
from __future__ import annotations

import argparse
import atexit
import ctypes as C
import functools
import json
import lzma
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

SEED = 20190901
ROWS_PER_BLOCK = 131072
TOTAL_BLOCKS = 64
METRIC = "TSV->ZDW encode GB/s (decode GB/s alongside) on synthetic analytics-hits-shaped TSV"


# --------------------------------------------------------------------------------------- generator
@functools.lru_cache(maxsize=1)
def _build_synth() -> Path:
    """The generator library: tools/libsynth_gen.so when it is up to date, else compiled once per process into a
    temporary directory that is removed at exit (the tree may be read-only)."""
    so = ROOT / "tools" / "libsynth_gen.so"
    src = ROOT / "tools" / "synth_gen.c"
    if not so.exists() or so.stat().st_mtime < src.stat().st_mtime:
        tmp = tempfile.mkdtemp(prefix="zdwsynth_")
        atexit.register(shutil.rmtree, tmp, ignore_errors=True)
        so = Path(tmp) / "libsynth_gen.so"
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-o", str(so), str(src)], check=True)
    return so


class Synth:
    def __init__(self):
        self.L = C.CDLL(str(_build_synth()))
        self.L.synth_profile_create.argtypes = [C.c_char_p, C.c_size_t, C.c_uint32]
        self.L.synth_profile_create.restype = C.c_void_p
        self.L.synth_block.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_size_t]
        self.L.synth_block.restype = C.c_size_t
        self.L.synth_max_row_bytes.argtypes = [C.c_void_p]
        self.L.synth_max_row_bytes.restype = C.c_uint32
        fixture = lzma.decompress((ROOT / "tests" / "golden" / "analytics-hits.sql.xz").read_bytes())
        self.desc = (ROOT / "tests" / "golden" / "analytics-hits.desc.sql").read_bytes()
        from zdw_b200.desc import parse_desc  # the product's own .desc.sql rules (host side)
        self.schema = parse_desc(self.desc)
        self.h = self.L.synth_profile_create(fixture, len(fixture), self.schema.ncols)
        if not self.h:
            raise RuntimeError("fixture does not parse")
        self.max_row = self.L.synth_max_row_bytes(self.h)

    def cap_for(self, rows: int) -> int:
        return rows * 4600 + self.max_row + (1 << 20)

    def block_into(self, block: int, rows: int, ptr: int, cap: int) -> int:
        n = self.L.synth_block(self.h, SEED, block, rows, C.c_void_p(ptr), cap)
        if n == 0:
            raise RuntimeError("synthetic block did not fit its buffer")
        return n


# --------------------------------------------------------------------------------------- helpers
def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi polled in the background.  It is started BEFORE the warm-up steps: its start-up (NVML init, first
    query) stalls kernel launches for some hundred milliseconds, which must not land in the timed region; only the
    samples whose timestamps fall inside [t_begin, t_end] are reported."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.p = None

    def start(self):
        if os.environ.get("ZDW_BENCH_NOCLOCK"):  # diagnostics only: a run without the poller reports no clocks
            return
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "250"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self, t_begin: float | None = None, t_end: float | None = None):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        import datetime
        sm, mx, reasons, sm_all = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            sm_all.append(clk)
            if t_begin is not None and not (t_begin - 0.05 <= ts <= t_end + 0.05):
                continue
            sm.append(clk)
            mx.append(cmax)
            for k, nme in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        if not sm and sm_all:  # region shorter than the polling period: fall back to every sample of the run
            sm, mx = sm_all, [max(sm_all)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# --------------------------------------------------------------------------------------- reference arm
def _ref_env():
    ref = ROOT / "oracle" / "_ref"
    env = dict(os.environ)
    env["PATH"] = f"{ref / 'nocomp'}:{env.get('PATH', '')}"
    return env


def _ref_roundtrip(workdir: Path, tsv_path: Path, desc: bytes):
    """One reference process: convertDWfile then unconvertDWfile on a shard. Returns (t_enc, t_dec, tsv_bytes)."""
    ref = ROOT / "oracle" / "_ref"
    (workdir / "x.desc.sql").write_bytes(desc)
    if tsv_path != workdir / "x.sql":
        os.symlink(tsv_path, workdir / "x.sql")
    env = _ref_env()
    t0 = time.perf_counter()
    subprocess.run([str(ref / "convertDWfile"), "-q", "x.sql"], cwd=workdir, env=env, check=True, capture_output=True)
    t1 = time.perf_counter()
    os.rename(workdir / "x.zdw.gz", workdir / "y.zdw")
    (workdir / "out").mkdir(exist_ok=True)
    subprocess.run([str(ref / "unconvertDWfile"), "-q", "-d", "out", "y.zdw"], cwd=workdir, env=env, check=True, capture_output=True)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, tsv_path.stat().st_size


def have_ref() -> bool:
    ref = ROOT / "oracle" / "_ref"
    return (ref / "convertDWfile").exists() and (ref / "unconvertDWfile").exists() and (ref / "nocomp" / "gzip").exists()



# --------------------------------------------------------------------------------------- parity gate (SURVEY 8(d))
def file_header_bytes(schema) -> bytes:
    """v11 file header without metadata: version, metadata length, names, types, char sizes (ConvertToZDW.cpp:673-737)."""
    hdr = (11).to_bytes(2, "little") + (0).to_bytes(4, "little")
    for nme in schema.names:
        hdr += (nme if isinstance(nme, bytes) else nme.encode("latin1")) + b"\0"
    return hdr + b"\0" + bytes(schema.types) + b"".join(int(c).to_bytes(2, "little") for c in schema.charsize)


def ref_encode_block(tsv_view, desc: bytes) -> bytes:
    """The unmodified compiled reference (oracle/_ref/convertDWfile, compressor stage = cat) on one block of rows.
    Returns its whole .zdw file (file header + one block)."""
    scratch = scratch_dir()
    try:
        with open(scratch / "x.sql", "wb") as f:
            f.write(tsv_view)
        (scratch / "x.desc.sql").write_bytes(desc)
        subprocess.run([str(ROOT / "oracle" / "_ref" / "convertDWfile"), "-q", "x.sql"], cwd=scratch, env=_ref_env(), check=True,
                       capture_output=True)
        return (scratch / "x.zdw.gz").read_bytes()
    finally:
        shutil.rmtree(scratch, ignore_errors=True)


def ref_decode_matches(image: bytes, expected_chunks) -> bool:
    """oracle/_ref/unconvertDWfile of `image` to a pipe, compared on the fly with the expected rows (an iterable of
    bytes-like chunks), so that no multi-GB TSV is ever held twice."""
    scratch = scratch_dir()
    try:
        (scratch / "x.zdw").write_bytes(image)
        p = subprocess.Popen([str(ROOT / "oracle" / "_ref" / "unconvertDWfile"), "-q", "-", "x.zdw"], cwd=scratch, env=_ref_env(),
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
        ok = True
        for chunk in expected_chunks:
            mv = memoryview(chunk).cast("B")
            pos = 0
            while ok and pos < len(mv):
                got = p.stdout.read(min(1 << 24, len(mv) - pos))
                if not got or got != mv[pos:pos + len(got)]:
                    ok = False
                pos += len(got)
            if not ok:
                break
        if ok and p.stdout.read(1):
            ok = False
        p.stdout.close()
        if not ok:
            p.kill()
        rc = p.wait()
        return ok and rc == 0
    finally:
        shutil.rmtree(scratch, ignore_errors=True)


def ref_parallel_step(synth: Synth, shard_rows: int, nproc: int, scratch: Path, inputs: list):
    """nproc independent reference processes, one shard each (the reference is single-threaded).
    Returns (enc_wall, dec_wall, total_tsv_bytes) with wall = slowest process."""
    res = [None] * nproc

    def work(i):
        wd = scratch / f"p{i}"
        if wd.exists():
            shutil.rmtree(wd)
        wd.mkdir(parents=True)
        res[i] = _ref_roundtrip(wd, inputs[i], synth.desc)

    with ThreadPoolExecutor(max_workers=nproc) as ex:
        list(ex.map(work, range(nproc)))
    return max(r[0] for r in res), max(r[1] for r in res), sum(r[2] for r in res)


def make_ref_inputs(synth: Synth, rows: int, nproc: int, scratch: Path):
    inputs = []
    cap = synth.cap_for(rows)
    buf = (C.c_uint8 * cap)()
    for i in range(nproc):
        n = synth.block_into(1000 + i, rows, C.addressof(buf), cap)
        p = scratch / f"shard{i}.sql"
        with open(p, "wb") as f:
            f.write(memoryview(buf)[:n])
        inputs.append(p)
    return inputs


def scratch_dir() -> Path:
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    return Path(tempfile.mkdtemp(prefix="zdwbench_", dir=base))


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    if not have_ref():
        # the oracle always exists: fall back to the C port when the compiled reference did not travel
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref binaries missing on this box"}))
        return 0
    synth = Synth()
    nproc = max(1, min(os.cpu_count() or 1, args.ref_procs))
    rows = args.ref_rows
    scratch = scratch_dir()
    try:
        inputs = make_ref_inputs(synth, rows, nproc, scratch)
        for _ in range(args.warmup):
            ref_parallel_step(synth, rows, nproc, scratch, inputs)
        te, td, tot = [], [], 0
        t_all0 = time.perf_counter()
        for _ in range(args.steps):
            e, d, b = ref_parallel_step(synth, rows, nproc, scratch, inputs)
            te.append(e)
            td.append(d)
            tot = b
        t_all = time.perf_counter() - t_all0
        enc = tot * args.steps / sum(te) / 1e9
        dec = tot * args.steps / sum(td) / 1e9
        sample = (f"{nproc} independent convertDWfile/unconvertDWfile processes (reference is single-threaded), one "
                  f"{rows}-row C4-shaped shard each ({tot / nproc / 1e6:.0f} MB), tmpfs, compressor stage replaced by cat")
        line = {
            "impl": "reference", "metric": METRIC, "value": enc, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args, note="bounded sample per step, see cpu_baseline.sample"),
            "decode": {"value": dec, "unit": "GB/s"},
            "cpu_baseline": {"value": enc, "decode_value": dec, "unit": "GB/s", "cores": nproc, "kind": "reference", "sample": sample},
            "e2e": {"value": enc, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "decode_value": dec},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
    finally:
        shutil.rmtree(scratch, ignore_errors=True)
    return 0


def workload_config(args, note=None):
    cfg = {"workload": (f"C4 synthetic analytics-hits-shaped TSV: 2086 columns (256 populated), {args.blocks} blocks x "
                        f"{args.rows_per_block} rows, seed {SEED}, block-sharded over {args.gpus} GPU(s)"),
           "blocks": args.blocks, "rows_per_block": args.rows_per_block, "parallelism": f"block-shard x{args.gpus}", "lanes_per_gpu": getattr(args, "lanes", 1),
           "l2": "inputs larger than L2 (every block is ~0.5 GB and is read once per pass)"}
    if note:
        cfg["note"] = note
    if getattr(args, "reduced_from", None):
        cfg["reduced"] = f"host RAM too small for {args.reduced_from} blocks; ran {args.blocks}"
    return cfg


# --------------------------------------------------------------------------------------- CUDA arm
def cpu_baseline_sample(synth: Synth, rows: int):
    """Reference (oracle/_ref) on ONE core over one bounded shard; rank 0, N=1 only."""
    if not have_ref():
        return None
    scratch = scratch_dir()
    try:
        inputs = make_ref_inputs(synth, rows, 1, scratch)
        e, d, b = ref_parallel_step(synth, rows, 1, scratch, inputs)
        return {"value": b / e / 1e9, "decode_value": b / d / 1e9, "unit": "GB/s", "cores": 1, "kind": "reference",
                "sample": f"one {rows}-row C4-shaped shard ({b / 1e6:.0f} MB): convertDWfile {e:.2f} s, unconvertDWfile {d:.2f} s, "
                          "single process (the reference has no threads), tmpfs, compressor stage replaced by cat"}
    finally:
        shutil.rmtree(scratch, ignore_errors=True)


def other_configs(torch, dev, local):
    """BASELINE configs C2 / C3 (the reference's own fixtures) and a C5-shaped block (high-cardinality text), device
    resident on this GPU: best-of-5 CUDA-event times of one encode and one decode call, with the parity each config
    allows - C2 / C3: the encoded bytes equal the reference's golden .zdw; C5: the decoded rows equal the input.
    These are parity-test cases (tests/), timed here so that the driver's record holds them too."""
    from zdw_b200 import Context
    from zdw_b200.desc import parse_desc
    out = []
    g = ROOT / "tests" / "golden"
    ctx = Context(local)
    ctx.set_stream(torch.cuda.current_stream(dev).cuda_stream)

    def time_call(fn):
        best = None
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None or ms < best else best
        return best, r

    def one(name, tsv, types, golden_block):
        t = torch.empty(len(tsv) + 64, dtype=torch.uint8, device=dev)
        t[:len(tsv)].copy_(torch.frombuffer(bytearray(tsv), dtype=torch.uint8))
        torch.cuda.synchronize(dev)
        enc = lambda: ctx.encode_block(types, t.data_ptr(), len(tsv), input_on_device=True, output_on_device=True)
        blk = enc()
        z = torch.empty(blk.length + 64, dtype=torch.uint8, device=dev)
        _d2d(torch, z, blk.dev_ptr, blk.length)
        dec = lambda: ctx.decode_block(types, z.data_ptr(), blk.length, input_on_device=True, output_on_device=True)
        d = dec()
        back = torch.empty(d.length, dtype=torch.uint8, device=dev)
        _d2d(torch, back, d.dev_ptr, d.length)
        roundtrip = d.length == len(tsv) and bool(torch.equal(back, t[:len(tsv)]))
        vs_golden = None
        if golden_block is not None:
            vs_golden = bytes(z[:blk.length].cpu().numpy().tobytes()) == golden_block
        e_ms, _ = time_call(enc)
        d_ms, _ = time_call(dec)
        out.append({"config": name, "tsv_bytes": len(tsv), "zdw_bytes": int(blk.length), "rows": int(blk.nrows),
                    "encode_ms": round(e_ms, 3), "decode_ms": round(d_ms, 3), "encode_gbs": round(len(tsv) / e_ms / 1e6, 2),
                    "decode_gbs": round(len(tsv) / d_ms / 1e6, 2), "zdw_equals_reference_golden": vs_golden,
                    "roundtrip_bit_exact": roundtrip, "timing": "device resident, best of 5, CUDA events"})

    for label, name in (("C2 movie_tickets (reference fixture)", "movie_tickets"), ("C3 analytics-hits (reference fixture)", "analytics-hits")):
        tsv = lzma.decompress((g / f"{name}.sql.xz").read_bytes())
        sch = parse_desc((g / f"{name}.desc.sql").read_bytes())
        gz = g / f"{name}.zdw"
        golden = gz.read_bytes() if gz.exists() else lzma.decompress((g / f"{name}.zdw.xz").read_bytes())
        # the golden files are v9 / v10: the block bytes follow their file header (no metadata section before v11)
        hdr_len = 2 + sum(len(n.encode("latin1")) + 1 for n in sch.names) + 1 + 3 * sch.ncols
        one(label, tsv, sch.types, golden[hdr_len:])
    import c5_check
    sch5 = parse_desc(c5_check.DESC)
    one("C5 high-cardinality text, 1 000 000 rows (2 M unique 65-byte strings, one block)", c5_check.make_rows(1_000_000), sch5.types, None)
    ctx.close()
    return out


def _parse_cpulist(text: str):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_node(torch, index: int):
    """Pins this process to the CPUs of the NUMA node the GPU hangs off (sysfs local_cpulist), so that the pinned host
    buffers of the e2e leg are allocated and first touched next to the GPU's PCIe root.  Best effort; returns a note."""
    try:
        pr = torch.cuda.get_device_properties(index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        cpus = _parse_cpulist(Path(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read_text())
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "unchanged (no local cpulist)"
        os.sched_setaffinity(0, cpus)
        node = Path(f"/sys/bus/pci/devices/{bdf}/numa_node").read_text().strip()
        return f"numa node {node} of GPU {bdf}: {len(cpus)} cpus"
    except Exception as ex:  # noqa: BLE001
        return f"unchanged ({type(ex).__name__})"


DUMP_ELEMENTS = 15 << 20  # float32 samples over all dumped arrays: 60 MiB


class _DeviceBytes:
    """n bytes at a device address, for torch.as_tensor (no copy, no stream synchronisation)."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 3, "stream": None}


class OutputSampler:
    """--dump-outputs.  Before the timed steps: seeded positions into every block's result (from its length in the untimed
    pass) and a buffer for the bytes there, both on the device.  In the last timed step: each call enqueues one gather
    of those positions on its lane's stream, before the lane's next call reuses the result buffer.  After the timed
    steps: the samples go to the host and into DIR/<name>.npy (float32), the per-block numbers into <name>_blocks.npy."""

    def __init__(self, torch, dev, block_ids, lengths: dict, per_block: int):
        self.torch, self.dev, self.block_ids, self.per_block = torch, dev, block_ids, per_block
        self.lengths = {name: list(ns) for name, ns in lengths.items()}
        self.idx = {name: [self._positions(name, j, n) for j, n in enumerate(ns)] for name, ns in lengths.items()}
        self.buf = {name: [torch.empty(len(i), dtype=torch.uint8, device=dev) for i in idx] for name, idx in self.idx.items()}
        self.numbers = {name: [None] * len(ns) for name, ns in lengths.items()}

    def _positions(self, name: str, j: int, n: int):
        import numpy as np
        if n <= self.per_block:
            idx = np.arange(n)
        else:
            seed = [SEED, self.block_ids[j], sorted(self.lengths).index(name)]
            idx = np.sort(np.random.default_rng(seed).integers(0, n, self.per_block))
        return self.torch.from_numpy(idx).to(self.dev)

    def take(self, stream, name: str, j: int, ptr: int, n: int, numbers):
        torch = self.torch
        self.numbers[name][j] = numbers
        if n != self.lengths[name][j]:  # a result longer or shorter than in the untimed pass: positions drawn here
            self.lengths[name][j] = n
            self.idx[name][j] = self._positions(name, j, n)
            self.buf[name][j] = torch.empty(len(self.idx[name][j]), dtype=torch.uint8, device=self.dev)
        view = torch.as_tensor(_DeviceBytes(ptr, n), device=self.dev)
        with torch.cuda.stream(stream):
            torch.index_select(view, 0, self.idx[name][j], out=self.buf[name][j])

    def write(self, out_dir: str, prefix: str):
        import numpy as np
        os.makedirs(out_dir, exist_ok=True)
        for name, bufs in self.buf.items():
            np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), np.concatenate([b.cpu().numpy() for b in bufs]).astype(np.float32))
            np.save(os.path.join(out_dir, f"{prefix}{name}_blocks.npy"), np.array(self.numbers[name], dtype=np.float64))


def run_cuda(args):
    import torch

    from zdw_b200 import Context
    from zdw_b200.capi import load_library

    rank, world, local = dist_env()
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = bind_to_gpu_node(torch, local)  # before any pinned allocation: first touch decides the NUMA node
    L = load_library()
    synth = Synth()
    types = synth.schema.types

    # ---- shard: whole blocks, contiguous ranges, in file order
    nb = args.blocks
    avail = _mem_available()
    need = 2.3 * nb / world * synth.cap_for(args.rows_per_block)
    if avail and need > avail:  # not enough host RAM for the named workload: shrink it and say so
        nb = max(world, int(nb * avail / need))
        args.reduced_from = args.blocks
        args.blocks = nb
    from zdw_b200.shard import block_range
    my_blocks = list(block_range(rank, world, nb))
    rows = args.rows_per_block

    # ---- host (pinned) inputs
    cap = synth.cap_for(rows)
    host_ptrs, host_lens = [], []
    pinned = True
    for _ in my_blocks:
        p = L.zdwb_host_alloc(cap)
        if not p:
            pinned = False
            break
        host_ptrs.append(p)
    if not pinned:  # fall back to pageable memory (e2e gets slower; recorded in the JSON line)
        for p in host_ptrs:
            L.zdwb_host_free(p)
        keep = [(C.c_uint8 * cap)() for _ in my_blocks]
        host_ptrs = [C.addressof(k) for k in keep]
    with ThreadPoolExecutor(max_workers=max(1, min(len(my_blocks), (os.cpu_count() or 2) // max(1, world), 16))) as ex:
        host_lens = list(ex.map(lambda ib: synth.block_into(ib[1], rows, host_ptrs[ib[0]], cap), list(enumerate(my_blocks))))
    tsv_bytes = sum(host_lens)

    ctx = Context(local)
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)

    # ---- device-resident inputs
    dev_tsv = []
    for p, n in zip(host_ptrs, host_lens):
        t = torch.empty(n + 64, dtype=torch.uint8, device=dev)
        arr = (C.c_uint8 * n).from_address(p)
        t[:n].copy_(torch.frombuffer(arr, dtype=torch.uint8), non_blocking=False)
        dev_tsv.append(t)
    torch.cuda.synchronize(dev)

    # ---- one untimed pass: produce the ZDW blocks the decoder will read, and keep host copies for e2e decode
    dev_zdw, zdw_lens, host_zdw = [], [], []
    for t, n in zip(dev_tsv, host_lens):
        blk = ctx.encode_block(types, t.data_ptr(), n, input_on_device=True, output_on_device=True)
        z = torch.empty(blk.length + 64, dtype=torch.uint8, device=dev)
        _d2d(torch, z, blk.dev_ptr, blk.length)
        dev_zdw.append(z)
        zdw_lens.append(blk.length)
    torch.cuda.synchronize(dev)
    zdw_bytes = sum(zdw_lens)
    for z, n in zip(dev_zdw, zdw_lens):
        host_zdw.append(z[:n].cpu().numpy().tobytes())

    # Blocks are independent, so RES_LANES contexts (one host thread + stream each) take the rank's blocks round-robin:
    # the host-side bookkeeping of one block (metadata read-backs, launch preparation) overlaps the kernels of another.
    # Every lane's stream is forked from / joined back into `stream`, so CUDA events on `stream` bracket all of it.
    res_lanes = [ctx]
    res_streams = [stream]
    for _ in range(max(1, args.lanes) - 1):
        ls = torch.cuda.Stream(device=dev)
        c2 = Context(local)
        c2.set_stream(ls.cuda_stream)
        res_lanes.append(c2)
        res_streams.append(ls)
    res_pool = ThreadPoolExecutor(max_workers=len(res_lanes))

    def _res_pass(fn, items):
        if len(res_lanes) == 1:
            for it in items:
                fn(ctx, it)
            return
        fork = torch.cuda.Event()
        fork.record(stream)
        for ls in res_streams[1:]:
            ls.wait_event(fork)

        def work(k):
            torch.cuda.set_device(dev)
            for j in range(k, len(items), len(res_lanes)):
                fn(res_lanes[k], items[j])
        list(res_pool.map(work, range(len(res_lanes))))
        for ls in res_streams[1:]:
            join = torch.cuda.Event()
            join.record(ls)
            stream.wait_event(join)

    enc_items = list(zip(dev_tsv, host_lens))
    dec_items = list(zip(dev_zdw, zdw_lens))

    # --dump-outputs: the samples of all ranks together stay within DUMP_ELEMENTS
    sampler_out = None
    if args.dump_outputs:
        sampler_out = OutputSampler(torch, dev, my_blocks, {"encode_zdw": zdw_lens, "decode_tsv": host_lens},
                                    DUMP_ELEMENTS // 2 // max(1, nb))
        torch.cuda.synchronize(dev)
    lane_stream = {id(c): s for c, s in zip(res_lanes, res_streams)}

    def encode_pass(sample=None):
        def one(c, j):
            t, n = enc_items[j]
            blk = c.encode_block(types, t.data_ptr(), n, input_on_device=True, output_on_device=True)
            if sample is not None:
                sample.take(lane_stream[id(c)], "encode_zdw", j, blk.dev_ptr, blk.length, (blk.length, blk.nrows, blk.longest_line))
        _res_pass(one, range(len(enc_items)))

    def decode_pass(sample=None):
        def one(c, j):
            z, n = dec_items[j]
            d = c.decode_block(types, z.data_ptr(), n, input_on_device=True, output_on_device=True)
            if sample is not None:
                sample.take(lane_stream[id(c)], "decode_tsv", j, d.dev_ptr, d.length, (d.length, d.nrows, d.line_length))
        _res_pass(one, range(len(dec_items)))

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- parity gate (SURVEY 8(d) "parity gate for every timing"): no number is printed unless it holds.
    #  (0) decode(encode(block 0)) == block 0 on the device;
    #  (a) every rank: the CUDA-encoded bytes of its first and last block == what the unmodified compiled reference
    #      (oracle/_ref/convertDWfile) writes for the same rows;
    #  (b) those blocks of ALL ranks, gathered on rank 0 and stitched in file order (isLast, cumulative longestLine:
    #      ConvertToZDW.cpp:841-842,965), go through the reference's unconvertDWfile and must come back as the source rows.
    rt = ctx.decode_block(types, dev_zdw[0].data_ptr(), zdw_lens[0], input_on_device=True, output_on_device=True)
    back = torch.empty(rt.length, dtype=torch.uint8, device=dev)
    _d2d(torch, back, rt.dev_ptr, rt.length)
    if rt.length != host_lens[0] or not torch.equal(back, dev_tsv[0][:host_lens[0]]):
        raise SystemExit("parity gate failed: decode(encode(block 0)) != block 0")
    del back
    parity = {"zdw_vs_ref": None, "tsv_vs_ref": None, "blocks": 0, "self_roundtrip": True}
    if args.no_parity:
        parity["note"] = "--no-parity: reference comparison skipped (diagnostic run, not a bench value)"
    elif not have_ref():
        parity["note"] = "oracle/_ref missing on this box: only the device round trip was checked"
    else:
        from zdw_b200.shard import stitch_blocks
        hdr = file_header_bytes(synth.schema)
        check = sorted({0, len(my_blocks) - 1})

        def _vs_ref(k):
            view = (C.c_uint8 * host_lens[k]).from_address(host_ptrs[k])
            ref_file = ref_encode_block(view, synth.desc)
            return ref_file[:len(hdr)] == hdr and ref_file[len(hdr):] == host_zdw[k]
        with ThreadPoolExecutor(max_workers=len(check)) as ex:
            zdw_ok = all(ex.map(_vs_ref, check))
        mine = [(my_blocks[k], host_zdw[k]) for k in check]
        gathered = [mine]
        if world > 1:
            import torch.distributed as dist
            gloo = dist.new_group(backend="gloo")
            gathered = [None] * world if rank == 0 else None
            dist.gather_object(mine, gathered, dst=0, group=gloo)
            flag = torch.tensor([1 if zdw_ok else 0], dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=gloo)
            zdw_ok = bool(flag.item())
        tsv_ok = True
        if rank == 0:
            allb = sorted(x for part in gathered for x in part)
            image = stitch_blocks(hdr, [b for _, b in allb])

            def _expected():
                scratch_buf = (C.c_uint8 * cap)()
                for bid, _ in allb:
                    m = synth.block_into(bid, rows, C.addressof(scratch_buf), cap)
                    yield memoryview(scratch_buf)[:m]
            tsv_ok = ref_decode_matches(image, _expected())
            parity.update({"zdw_vs_ref": zdw_ok, "tsv_vs_ref": tsv_ok, "blocks": len(allb),
                           "checked": ("first and last block of every rank: CUDA bytes == oracle/_ref/convertDWfile bytes; the "
                                       f"{len(allb)} blocks stitched in file order on rank 0 -> oracle/_ref/unconvertDWfile == source rows")})
        if world > 1:
            flag = torch.tensor([1 if (zdw_ok and tsv_ok) else 0], dtype=torch.int32)
            dist.broadcast(flag, src=0, group=gloo)
            if not flag.item():
                raise SystemExit("parity gate failed: CUDA output differs from the reference (see rank 0)")
        elif not (zdw_ok and tsv_ok):
            raise SystemExit(f"parity gate failed: zdw_vs_ref={zdw_ok} tsv_vs_ref={tsv_ok}")

    sampler = ClockSampler(local)
    sampler.start()
    t_sampler = time.time()
    for _ in range(args.warmup):
        encode_pass()
        decode_pass()
    barrier()
    while time.time() - t_sampler < 2.0:  # let the poller get past its start-up before timing starts (extra warm-up)
        encode_pass()
        decode_pass()
    barrier()

    launches0 = sum(c.kernel_launches() for c in res_lanes)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    enc_ms, dec_ms = [], []
    barrier()
    t_wall0 = time.perf_counter()
    t_epoch0 = time.time()
    for step in range(args.steps):
        sample = sampler_out if step == args.steps - 1 else None
        ev[0].record(stream)
        encode_pass(sample)
        ev[1].record(stream)
        decode_pass(sample)
        ev[2].record(stream)
        ev[2].synchronize()
        enc_ms.append(ev[0].elapsed_time(ev[1]))
        dec_ms.append(ev[1].elapsed_time(ev[2]))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = sum(c.kernel_launches() for c in res_lanes) - launches0
    clocks = sampler.stop(t_epoch0, time.time())
    if sampler_out is not None:
        sampler_out.write(args.dump_outputs, f"rank{rank}_" if world > 1 else "")

    # ---- end to end through the C ABI with HOST buffers (H2D + kernels + D2H inside the timed region).  Blocks are
    # independent, so E2E_LANES contexts (one host thread + stream each) work on different blocks at the same time: the
    # PCIe copy of one block overlaps the kernels of another.  Every call is a plain zdwb_encode_block /
    # zdwb_decode_block with host pointers; the ZDW blocks / TSV rows come back in pinned host memory.
    lanes = [Context(local) for _ in range(max(1, args.e2e_lanes))]
    if args.copy_gate is not None:  # A/B of the library's copy gate (default: on)
        for c in lanes:
            c.set_tuning("copy_gate", args.copy_gate)
    for kv in args.e2e_tune:  # A/B of any other knob of the library in the e2e leg (diagnostic)
        k, v = kv.split("=")
        for c in lanes:
            c.set_tuning(k, int(v))
    pool = ThreadPoolExecutor(max_workers=len(lanes))

    def _run_lanes(fn, items):
        def work(k):
            tot = 0
            for j in range(k, len(items), len(lanes)):
                tot += fn(lanes[k], items[j])
            return tot
        return sum(pool.map(work, range(len(lanes))))

    def e2e_encode_pass():
        return _run_lanes(lambda c, it: L_encode_host(c, types, it[0], it[1]), list(zip(host_ptrs, host_lens)))

    # the ZDW blocks the e2e decode reads: pinned like the TSV inputs (a pageable source makes the driver stage the copy
    # under its own lock, which holds up the other contexts' copies); plain buffers only if pinning fails
    e2e_dec_blocks, dec_keep, dec_pinned = [], [], []
    for zb in host_zdw[:max(1, args.e2e_decode_blocks)]:  # (the rank's blocks; repeated below when it has fewer than 24)
        p = L.zdwb_host_alloc(len(zb)) if pinned else None
        if p:
            C.memmove(p, zb, len(zb))
            dec_pinned.append(p)
        else:
            buf = (C.c_uint8 * len(zb)).from_buffer_copy(zb)
            dec_keep.append(buf)
            p = C.addressof(buf)
        e2e_dec_blocks.append((p, len(zb)))

    def e2e_decode_pass(items):
        return _run_lanes(lambda c, it: L_decode_host(c, types, it[0], it[1]), items)

    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    e2e_encode_pass()
    barrier()
    t0 = time.perf_counter()
    d2h_enc = 0
    for _ in range(e2e_steps):
        d2h_enc = e2e_encode_pass()
    torch.cuda.synchronize(dev)
    t_e2e_enc = (time.perf_counter() - t0) / e2e_steps
    # every rank decodes at least 24 blocks (its own, over again if need be) so that the lanes have something to overlap;
    # a context writes its first three results to pageable memory (pinning costs more than it saves for a short-lived
    # context), so four blocks per lane are warm-up
    reps = max(1, -(-24 // max(1, len(e2e_dec_blocks))))
    e2e_dec_items = e2e_dec_blocks * reps
    e2e_decode_pass((e2e_dec_blocks * 4)[:4 * len(lanes)])
    barrier()
    t0 = time.perf_counter()
    d2h_dec = e2e_decode_pass(e2e_dec_items)
    torch.cuda.synchronize(dev)
    t_e2e_dec = time.perf_counter() - t0
    launches_e2e = sum(c.kernel_launches() for c in lanes)
    # plain pinned-host <-> device copies of one block by EVERY rank at the same time (between barriers): the link ceiling
    # the e2e numbers sit under - at N > 1 the ranks share the host's memory and PCIe root ports, so the per-rank rate
    # is lower than a rank's rate when it copies alone
    pcie = {}
    try:
        hp = torch.empty(host_lens[0], dtype=torch.uint8).pin_memory()
        dp = torch.empty(host_lens[0], dtype=torch.uint8, device=dev)
        for name, (dst, src) in (("h2d_gbs", (dp, hp)), ("d2h_gbs", (hp, dp))):
            dst.copy_(src, non_blocking=True)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            e1.record(stream)
            e1.synchronize()
            pcie[name] = 4 * host_lens[0] / (e0.elapsed_time(e1) / 1e3) / 1e9
            barrier()
        del hp, dp
    except Exception as ex:  # noqa: BLE001
        pcie = {"error": str(ex)}
    link = torch.tensor([pcie.get("h2d_gbs", 0.0), pcie.get("d2h_gbs", 0.0)], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(link, op=dist.ReduceOp.SUM)  # the box's concurrent copy rate, all ranks together
    link_h2d, link_d2h = [float(x) for x in link.tolist()]
    pool.shutdown()
    for c in lanes:
        c.close()
    for p in dec_pinned:
        L.zdwb_host_free(p)

    # ---- instrumented step: per-kernel CUDA-event times for the roofline
    # (one context walks every block of the rank, so the launch count per kernel equals the number of blocks)
    ctx.set_tuning("kernel_timing", 1)
    ctx.kernel_times()
    for it in enc_items:
        ctx.encode_block(types, it[0].data_ptr(), it[1], input_on_device=True, output_on_device=True)
    kt_enc = ctx.kernel_times()
    for it in dec_items:
        ctx.decode_block(types, it[0].data_ptr(), it[1], input_on_device=True, output_on_device=True)
    kt_dec = ctx.kernel_times()
    ctx.set_tuning("kernel_timing", 0)

    # ---- reduce over ranks: time = max, bytes = sum
    enc_t = sum(enc_ms) / 1e3
    dec_t = sum(dec_ms) / 1e3
    if os.environ.get("ZDW_BENCH_DEBUG"):
        print(f"[rank {rank}] enc_ms={enc_ms} dec_ms={dec_ms} kt_dec={sorted(kt_dec.items(), key=lambda kv: -kv[1][1])[:4]}",
              file=sys.stderr, flush=True)
    vals = torch.tensor([enc_t, dec_t, t_e2e_enc, t_e2e_dec, t_wall], dtype=torch.float64, device=dev)
    sums = torch.tensor([tsv_bytes, zdw_bytes, float(d2h_enc), float(d2h_dec), float(launches),
                         float(sum(host_lens[:len(e2e_dec_blocks)]) * reps)], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    enc_t, dec_t, t_e2e_enc, t_e2e_dec, t_wall = [float(x) for x in vals.tolist()]
    tot_tsv, tot_zdw, d2h_enc_all, d2h_dec_all, launches_all, e2e_dec_tsv = [float(x) for x in sums.tolist()]

    if rank == 0:
        peak, peak_src = measured_peak()
        enc_gbs = tot_tsv * args.steps / enc_t / 1e9
        dec_gbs = tot_tsv * args.steps / dec_t / 1e9
        nblk = len(my_blocks)
        alg_bytes_block = (tsv_bytes + zdw_bytes) / nblk  # SURVEY 8(d): B_enc = B_dec = TSV + ZDW bytes of a block

        def roof(kt, traffic_key):
            if not kt:
                return None
            name, (cnt, ms) = max(kt.items(), key=lambda kv: kv[1][1])
            per_launch_s = ms / 1e3 / nblk  # this kernel's time per block (it is launched once per block)
            ach = alg_bytes_block / per_launch_s / 1e9
            total_ms = sum(v[1] for v in kt.values())
            return {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "peak_source": peak_src, "traffic": _traffic(name),
                    "algorithmic_bytes_per_launch": alg_bytes_block, "launch_ms": per_launch_s * 1e3,
                    "launches_per_block": cnt / nblk,
                    "share_of_step": ms / total_ms if total_ms else None,
                    "kernels_ms_per_block": {k: round(v[1] / nblk, 4) for k, v in sorted(kt.items(), key=lambda kv: -kv[1][1])},
                    "timed": "instrumented step (CUDA events around every launch) right after the timed steps"}

        line = {
            "metric": METRIC, "value": enc_gbs, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * (enc_t + dec_t) / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(args),
            "encode": {"value": enc_gbs, "unit": "GB/s", "ms_per_step": 1e3 * enc_t / args.steps,
                       "pipeline_frac_of_hbm_peak": (tot_tsv + tot_zdw) * args.steps / enc_t / 1e9 / (peak * world)},
            "decode": {"value": dec_gbs, "unit": "GB/s", "ms_per_step": 1e3 * dec_t / args.steps,
                       "pipeline_frac_of_hbm_peak": (tot_tsv + tot_zdw) * args.steps / dec_t / 1e9 / (peak * world),
                       "roofline": roof(kt_dec, "decode")},
            "roofline": roof(kt_enc, "encode"),
            "e2e": {"value": tot_tsv / t_e2e_enc / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(tot_tsv),
                    "d2h_bytes_per_step": int(d2h_enc_all), "pinned_host_input": pinned, "cpu_affinity": affinity, "lanes": args.e2e_lanes,
                    "pcie_copy_gbs": pcie,
                    # all ranks copying at once: what the host side of the box delivers; the e2e legs as a fraction of it
                    # (encode moves its bytes host -> device, decode device -> host)
                    "link_concurrent_gbs": {"h2d": link_h2d, "d2h": link_d2h},
                    "frac_of_link": (tot_tsv / t_e2e_enc / 1e9) / link_h2d if link_h2d else None,
                    "decode_frac_of_link": (e2e_dec_tsv / t_e2e_dec / 1e9) / link_d2h if link_d2h else None,
                    "decode_value": e2e_dec_tsv / t_e2e_dec / 1e9, "decode_blocks_timed": len(e2e_dec_items), "pinned_decode_input": bool(dec_pinned) and not dec_keep,
                    "decode_d2h_bytes": int(d2h_dec_all)},
            "gpu_launches": int(launches_all),
            "dump_outputs": args.dump_outputs,
            "parity": parity,
            "clocks": clocks,
            "tsv_bytes": int(tot_tsv), "zdw_bytes": int(tot_zdw),
            "wall_s_timed_region": t_wall,
        }
        if world == 1 and not args.no_configs:
            try:
                line["configs"] = other_configs(torch, dev, local)
            except Exception as ex:  # noqa: BLE001
                line["configs"] = {"error": f"{type(ex).__name__}: {ex}"}
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline_sample(synth, args.cpu_rows)
            line["cpu_baseline"] = cb if cb else {"value": None, "unit": "GB/s", "cores": 0, "kind": "reference",
                                                  "sample": "oracle/_ref missing on this box"}
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return 0


def _mem_available():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024 // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    except OSError:
        pass
    return None


def _traffic(kernel: str):
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(kernel)
        except Exception:
            return None
    return None


def _d2d(torch, dst_tensor, src_ptr: int, n: int):
    """device->device copy from a raw pointer into a torch tensor (plain cudaMemcpyAsync on torch's stream)."""
    cudart = _cudart()
    rc = cudart.cudaMemcpyAsync(C.c_void_p(dst_tensor.data_ptr()), C.c_void_p(src_ptr), C.c_size_t(n), 3,
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))
    if rc != 0:
        raise RuntimeError(f"cudaMemcpyAsync failed: {rc}")
    torch.cuda.current_stream().synchronize()


_CUDART = None


def _cudart():
    global _CUDART
    if _CUDART is None:
        for name in ("libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
            try:
                _CUDART = C.CDLL(name)
                break
            except OSError:
                continue
        _CUDART.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    return _CUDART


def L_decode_host(ctx, types, ptr: int, n: int) -> int:
    """Host ZDW block in, host TSV out (left in the context's pinned buffer), no copies through Python."""
    from zdw_b200 import capi
    tarr = (C.c_uint8 * len(types))(*types)
    sch = capi._Schema(len(types), C.cast(tarr, C.POINTER(C.c_uint8)))
    o = capi._DecOpts()
    o.at_end_of_file = 1
    o.separator = 9
    o.rownum_pos = -1
    out = capi._RowsOut()
    rc = ctx._L.zdwb_decode_block(ctx._h, C.byref(sch), C.c_void_p(ptr), n, C.byref(o), C.byref(out))
    if rc:
        raise RuntimeError(ctx.last_error())
    return int(out.len)


def L_encode_host(ctx, types, ptr: int, n: int) -> int:
    """Host pointer in, host bytes out, without copying the input through Python."""
    from zdw_b200 import capi
    tarr = (C.c_uint8 * len(types))(*types)
    sch = capi._Schema(len(types), C.cast(tarr, C.POINTER(C.c_uint8)))
    o = capi._EncOpts(0, 0, 0, 0, 0, 0, 0, 0, 0)
    out = capi._BlockOut()
    rc = ctx._L.zdwb_encode_block(ctx._h, C.byref(sch), C.c_void_p(ptr), n, C.byref(o), C.byref(out))
    if rc:
        raise RuntimeError(ctx.last_error())
    return int(out.len)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--blocks", type=int, default=TOTAL_BLOCKS)
    ap.add_argument("--rows-per-block", type=int, default=ROWS_PER_BLOCK)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-decode-blocks", type=int, default=48)
    ap.add_argument("--lanes", type=int, default=4, help="contexts (host thread + stream) that share the rank's blocks in the device-resident leg")
    ap.add_argument("--e2e-lanes", type=int, default=3, help="contexts (host thread + stream) that overlap copies and kernels in the e2e leg")
    ap.add_argument("--copy-gate", type=int, default=None, help="0 / 1: large copies of the e2e contexts take turns (library default: 1)")
    ap.add_argument("--e2e-tune", action="append", default=[], help="name=value tuning knob for the e2e contexts (diagnostic A/B)")
    ap.add_argument("--cpu-rows", type=int, default=131072, help="rows of the bounded cpu_baseline sample")
    ap.add_argument("--ref-rows", type=int, default=32768, help="rows per process per step of --impl reference")
    ap.add_argument("--ref-procs", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C2 / C3 / C5 timings of the N=1 line")
    ap.add_argument("--no-parity", action="store_true", help="skip the comparison with oracle/_ref (diagnostic runs only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/*.npy: a seeded sample of every block's ZDW bytes "
                         "and decoded TSV bytes (float32, %d MiB in all) and per block its length, rows and longest "
                         "line (float64); the timed calls only enqueue a gather of positions drawn beforehand" % (DUMP_ELEMENTS * 4 >> 20))
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "cuda":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())
