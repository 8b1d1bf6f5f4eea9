"""Reading ZDW files into typed device columns.

  header, blocks = read_columns("hits.zdw.gz", ["ip", "date_time"])
  blocks[0].values        # (2, nrows) int64 CUDA tensor: codes of the two text columns
  blocks[0].strings(0)    # their texts on the host

  header, table = read_table("hits.zdw.gz", ["ip", "date_time"])
  table.values            # (2, total_rows) int64 CUDA tensor: codes into each column's file-wide dictionary
  table.strings(0)        # the texts of the first column on the host

The file header (version, metadata, column names, types, char sizes) is read on the host; every block goes through
zdwb_decode_columns on the GPU (see capi.ColumnBlock for what the values mean).  read_table then merges every text-like
column's block dictionaries into one with zdwb_merge_codes.
"""
from __future__ import annotations

import bz2
import gzip
import lzma
import os
import struct
from dataclasses import dataclass

from .capi import TEXT_LIKE_TYPES, ColumnBlock, Context, _strings


@dataclass
class FileHeader:
    version: int        # 9, 10 or 11 (the block layout is the same)
    metadata: dict      # {key: value} (str, latin-1), v11 only; empty for v9 / v10
    names: list         # column names (str, latin-1)
    types: list         # column type ids (include/zdw_b200.h)
    charsize: list      # varchar(N) / char(N) -> N, else 0
    length: int         # bytes of the header: the first block starts here


def read_header(image: bytes) -> FileHeader:
    """The file header of a ZDW v9 / v10 / v11 image (UnconvertFromZDW.cpp:1042-1200).  ValueError when it is not one."""
    if not isinstance(image, (bytes, bytearray)):
        image = bytes(image)
    n = len(image)
    if n < 2:
        raise ValueError("ZDW header: file too short")
    (version,) = struct.unpack_from("<H", image, 0)
    if version < 9 or version > 11:
        raise ValueError(f"ZDW header: version {version} is not supported (versions 9-11 are)")
    pos = 2
    metadata = {}
    if version >= 11:
        if n < pos + 4:
            raise ValueError("ZDW header: truncated metadata length")
        (ml,) = struct.unpack_from("<I", image, pos)
        pos += 4
        if n < pos + ml:
            raise ValueError("ZDW header: truncated metadata")
        block = bytes(image[pos:pos + ml]) + b"\0"
        pos += ml
        at = 0
        while at < ml:  # key\0value\0 ...
            z = block.index(b"\0", at)
            key, at = block[at:z], z + 1
            if at < ml:
                z = block.index(b"\0", at)
                value, at = block[at:z], z + 1
            else:
                value, at = b"", at + 1
            metadata[key.decode("latin1")] = value.decode("latin1")
    names = []
    while True:
        z = image.find(b"\0", pos)
        if z < 0:
            raise ValueError("ZDW header: truncated column names")
        if z == pos:
            pos += 1
            break
        names.append(bytes(image[pos:z]).decode("latin1"))
        pos = z + 1
    nc = len(names)
    if n < pos + 3 * nc:
        raise ValueError("ZDW header: truncated column types")
    types = list(image[pos:pos + nc])
    pos += nc
    charsize = list(struct.unpack_from(f"<{nc}H", image, pos))
    pos += 2 * nc
    return FileHeader(version, metadata, names, types, charsize, pos)


@dataclass
class ColumnTable:
    """A whole ZDW file as typed device columns (read_table): row k of `values` is file column columns[k].

    values      (K, total_rows) int64 CUDA tensor.  Integer and CHAR columns hold what ColumnBlock.values holds, the
                blocks' rows concatenated.  Text-like columns hold codes into that column's file-wide dictionary
                dicts[k] (-1 = no value): dense (every code 0 .. entries - 1 occurs), sorted bytewise so that codes
                compare like the strings, equal iff the strings are equal.
    dicts       per row of `values`: (dict, entry_off) for a text-like column - a uint8 CUDA tensor laid out as
                ColumnBlock.dict and an int64 CUDA tensor of entries + 1 offsets - and None for the other columns.
    columns     file column index of every row of `values`.
    block_rows  rows per block, in file order.
    """
    values: object
    dicts: list
    columns: list
    block_rows: list

    def strings(self, k: int) -> list:
        """The texts of row k of `values` (a text-like column) on the host: bytes per row, None for code -1."""
        if self.dicts[k] is None:
            raise ValueError(f"row {k} of the table is not a text-like column")
        return _strings(self.values[k], *self.dicts[k])


def _load(path) -> bytes:
    """The file's bytes, decompressed by suffix as the reference does (UnconvertFromZDW.cpp:235-256)."""
    p = os.fspath(path)
    if p.endswith(".gz"):
        with gzip.open(p, "rb") as f:
            return f.read()
    if p.endswith(".bz2"):
        with bz2.open(p, "rb") as f:
            return f.read()
    if p.endswith(".xz"):
        with lzma.open(p, "rb") as f:
            return f.read()
    if p.endswith(".zst"):
        raise ValueError(f"{p}: zstd-compressed ZDW files are not supported here (the standard library has no zstd); "
                         "decompress the file first")
    with open(p, "rb") as f:
        return f.read()


def _open(path_or_bytes, columns):
    """(image, header, file column indices of `columns`)"""
    if isinstance(path_or_bytes, (bytes, bytearray, memoryview)):
        image = bytes(path_or_bytes)
    else:
        image = _load(path_or_bytes)
    hdr = read_header(image)
    if columns is None:
        cols = list(range(len(hdr.names)))
    else:
        where = {nm: i for i, nm in enumerate(hdr.names)}
        missing = [nm for nm in columns if nm not in where]
        if missing:
            raise KeyError(f"no such column(s) in the file: {missing}")
        cols = [where[nm] for nm in columns]
    return image, hdr, cols


def _decode_blocks(ctx, image, hdr, cols) -> list:
    blocks = []
    pos = hdr.length
    while True:
        blk = ctx.decode_columns(hdr.types, image, cols, len(image) - pos, at_end_of_file=True, offset=pos)
        blocks.append(blk)
        pos += blk.consumed
        if blk.is_last:
            break
    return blocks


def read_columns(path_or_bytes, columns=None, device: int = 0) -> tuple[FileHeader, list[ColumnBlock]]:
    """Decodes every block of a ZDW file into typed device columns.  path_or_bytes: a path (.gz / .bz2 / .xz are
    decompressed) or the file image itself.  columns: column names in the order wanted, None = all.  Returns the header
    and one ColumnBlock per block, whose `values` rows follow `columns`."""
    image, hdr, cols = _open(path_or_bytes, columns)
    with Context(device) as ctx:
        blocks = _decode_blocks(ctx, image, hdr, cols)
    return hdr, blocks


def read_table(path_or_bytes, columns=None, device: int = 0) -> tuple[FileHeader, ColumnTable]:
    """Decodes a whole ZDW file into one ColumnTable: the inputs are those of read_columns.  Every block is decoded with
    zdwb_decode_columns; the codes of each text-like column are then merged over all blocks by one zdwb_merge_codes call
    into a file-wide dictionary, the other columns are the blocks' rows concatenated.
    Peak device memory: the decoded blocks (values and dictionaries of every block) and the table, plus, during the merge
    of one column, its scratch and outputs (include/zdw_b200.h): 4 bytes per entry of every block dictionary (they hold
    the strings of all columns, not only this one's), 88 bytes per referenced (block, entry) pair summed over the blocks,
    and the merged codes (8 bytes per row) and dictionary, which live until they are copied into the table."""
    import torch

    image, hdr, cols = _open(path_or_bytes, columns)
    with Context(device) as ctx:
        blocks = _decode_blocks(ctx, image, hdr, cols)
        block_rows = [b.nrows for b in blocks]
        total = sum(block_rows)
        values = torch.empty((len(cols), total), dtype=torch.int64, device=f"cuda:{device}")
        dicts = []
        for k, c in enumerate(cols):
            if hdr.types[c] in TEXT_LIKE_TYPES:
                m = ctx.merge_codes([(b.dict, b.entry_off, b.values[k]) for b in blocks])
                values[k].copy_(m.codes)
                dicts.append((m.dict, m.entry_off))
            else:
                values[k].copy_(torch.cat([b.values[k] for b in blocks]))
                dicts.append(None)
    return hdr, ColumnTable(values, dicts, cols, block_rows)
