"""Writing typed device columns as a ZDW file: the way back from read_table.

  header, table = read_table("hits.zdw.gz")
  keep = table.values[3] > 0                      # edit the table in torch ...
  table = ColumnTable(table.values[:, keep], table.dicts, table.columns, [int(keep.sum())])
  write_table("hits_filtered.zdw.gz", header, table)

Every block is rendered to TSV rows on the GPU by zdwb_render_columns and encoded by zdwb_encode_block, so a written file
is byte for byte what convertDWfile makes of the rendered text.  The file header is written on the host.
"""
from __future__ import annotations

import bz2
import gzip
import lzma
import os
import struct

from .capi import Context
from .reader import ColumnTable, FileHeader


def _file_header(header: FileHeader, cols: list) -> bytes:
    """A v11 file header (ConvertToZDW.cpp:673-737) of the file columns `cols`, metadata keys in sorted order."""
    meta = b"".join(k.encode("latin1") + b"\0" + v.encode("latin1") + b"\0" for k, v in sorted(header.metadata.items()))
    out = struct.pack("<HI", 11, len(meta)) + meta
    out += b"".join(header.names[c].encode("latin1") + b"\0" for c in cols) + b"\0"
    out += bytes(header.types[c] for c in cols)
    out += b"".join(struct.pack("<H", header.charsize[c]) for c in cols)
    return out


def _open_out(path):
    """The output file, compressed by suffix as read_table reads it."""
    p = os.fspath(path)
    if p.endswith(".zst"):
        raise ValueError(f"{p}: zstd-compressed ZDW files are not supported here (the standard library has no zstd)")
    if p.endswith(".gz"):
        return gzip.open(p, "wb")
    if p.endswith(".bz2"):
        return bz2.open(p, "wb")
    if p.endswith(".xz"):
        return lzma.open(p, "wb")
    return open(p, "wb")


def write_table(path, header: FileHeader, table: ColumnTable, *, rows_per_block: int | None = None, device: int = 0) -> None:
    """Writes `table` as a ZDW v11 file.  Row k of table.values is file column header index table.columns[k]: names, types
    and char sizes come from `header` at those indices, so a projection writes a file of just those columns, in the
    table's order.  The metadata is header.metadata.  Blocks follow table.block_rows, or hold rows_per_block rows each
    (the last one the rest) when that is given.  path: .gz, .bz2 and .xz are compressed by the standard library, .zst is
    refused.  The writer waits for torch's current stream first, so cells computed there are final."""
    import torch

    cols = list(table.columns)
    K = len(cols)
    values = table.values
    if not isinstance(values, torch.Tensor) or not values.is_cuda or values.device.index != device:
        raise ValueError(f"write_table: values must be a tensor on cuda:{device}")
    if values.dtype != torch.int64 or values.dim() != 2 or values.shape[0] != K:
        raise ValueError(f"write_table: values must be a ({K}, rows) int64 tensor")
    if len(table.dicts) != K:
        raise ValueError(f"write_table: {len(table.dicts)} dicts for {K} columns")
    for c in cols:
        if not 0 <= c < len(header.names):
            raise ValueError(f"write_table: column index {c} is not in the header")
    for k, dd in enumerate(table.dicts):
        for t in (dd or ()):
            if not isinstance(t, torch.Tensor) or not t.is_cuda or t.device.index != device:
                raise ValueError(f"write_table: the dictionary of row {k} must be on cuda:{device}")
    total = values.shape[1]
    if total == 0:
        raise ValueError("write_table: the table has no rows (convertDWfile: Empty data file)")
    if rows_per_block is not None:
        if rows_per_block <= 0:
            raise ValueError("write_table: rows_per_block must be positive")
        sizes = [min(rows_per_block, total - s) for s in range(0, total, rows_per_block)]
    else:
        sizes = [int(b) for b in table.block_rows]
        if any(b <= 0 for b in sizes) or sum(sizes) != total:
            raise ValueError(f"write_table: block_rows {sizes[:8]}... must be positive and sum to the {total} rows")
    values = values.contiguous()
    types = [header.types[c] for c in cols]
    torch.cuda.current_stream(device).synchronize()
    with Context(device) as ctx, _open_out(path) as f:
        f.write(_file_header(header, cols))
        start = 0
        longest = 0
        for b, rows in enumerate(sizes):
            # the first row of the next block is rendered too: the reference reads it before it closes this block, and its
            # length counts for this block's longest line; encode_block stops after `rows` rows and writes isLast = 0
            end = start + rows + (1 if b + 1 < len(sizes) else 0)
            ptr, n = ctx.render_columns(types, values[:, start:end], table.dicts)
            blk = ctx.encode_block(types, ptr, n, input_on_device=True, prev_longest_line=longest, max_rows=rows)
            if blk.nrows != rows:
                raise RuntimeError(f"write_table: block {b} encoded {blk.nrows} rows instead of {rows}")
            f.write(blk.data)
            longest = blk.longest_line
            start += rows
