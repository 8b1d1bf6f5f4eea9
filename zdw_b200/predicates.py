"""Filters on the text columns of a ColumnTable, on the GPU: LIKE, IN and BETWEEN.

  hdr, t = read_table("hits.zdw.gz")
  keep = like(hdr, t, 5, b"%/checkout%") & between(hdr, t, 2, b"2024-03-01", b"2024-03-07 23:59:59")
  write_table("checkout.zdw.gz", hdr, ColumnTable(t.values[:, keep], t.dicts, t.columns, [int(keep.sum())]))

A column's dictionary holds each distinct string once, sorted bytewise, and its codes compare like the strings.  So each
predicate runs once per dictionary entry (zdwb_match_like, zdwb_find_strings) and then one gather or two integer
compares per row.  Code -1 stands for the column's null text: "" for text columns, "0.000000000000" for DECIMAL (the
text unconvertDWfile prints for it), and it matches as that text would.
"""
from __future__ import annotations

from .capi import TEXT_LIKE_TYPES, Context
from .reader import ColumnTable, FileHeader

DECIMAL = 11


def _text_column(header: FileHeader, table: ColumnTable, k: int):
    """(codes, dict, entry_off, null text) of row k of the table, after torch's current stream has finished."""
    import torch
    t = header.types[table.columns[k]]
    if t not in TEXT_LIKE_TYPES or table.dicts[k] is None:
        raise ValueError(f"row {k} of the table (file column {table.columns[k]}, type {t}) is not a text-like column")
    codes = table.values[k]
    torch.cuda.current_stream(codes.device).synchronize()
    dct, eo = table.dicts[k]
    return codes, dct, eo, (b"0.000000000000" if t == DECIMAL else b"")


def like(header: FileHeader, table: ColumnTable, k: int, pattern: bytes, *, escape: bytes | None = b"\\",
         ignore_case: bool = False):
    """Row k of table.values LIKE pattern (Context.match_like gives the rules: bytewise, '_' is one byte): a bool CUDA
    tensor with one flag per row."""
    codes, dct, eo, null = _text_column(header, table, k)
    with Context(codes.device.index) as ctx:
        flags = ctx.match_like(dct, eo, pattern, escape=escape, ignore_case=ignore_case, null_text=null)
    return flags[codes]  # code -1 takes the last flag, null_text's


def isin(header: FileHeader, table: ColumnTable, k: int, strings):
    """Row k of table.values IN strings (a sequence of bytes): a bool CUDA tensor with one flag per row."""
    import torch
    codes, dct, eo, null = _text_column(header, table, k)
    strings = [bytes(s) for s in strings]
    with Context(codes.device.index) as ctx:
        rank, found = ctx.find_strings(dct, eo, strings)
    flags = torch.zeros(eo.numel(), dtype=torch.bool, device=codes.device)  # entries + 1: the last one for code -1
    flags[rank[found]] = True
    flags[-1] = null in strings
    return flags[codes]


def between(header: FileHeader, table: ColumnTable, k: int, lo: bytes, hi: bytes):
    """Row k of table.values BETWEEN lo AND hi, both ends included, bytewise: a bool CUDA tensor with one flag per row.
    On a DATETIME column this is a date range.  lo > hi matches nothing."""
    import torch
    codes, dct, eo, null = _text_column(header, table, k)
    lo, hi = bytes(lo), bytes(hi)
    with Context(codes.device.index) as ctx:
        rank, found = ctx.find_strings(dct, eo, [lo, hi])
    # codes compare like their strings: lo <= s iff code >= rank(lo); s <= hi iff code < rank(hi) + found(hi)
    inside = (codes >= rank[0]) & (codes < rank[1] + found[1].long())
    return torch.where(codes < 0, torch.tensor(lo <= null <= hi, device=codes.device), inside)
