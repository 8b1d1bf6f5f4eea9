"""DATETIME and DECIMAL columns of a ColumnTable as numbers, on the GPU, and numbers back as text columns.

  hdr, t = read_table("movie_tickets.zdw")
  us, _ = to_datetime(hdr, t, 0)               # int64 microseconds since 1970-01-01
  cents, _ = to_decimal(hdr, t, 5, scale=2)    # int64 revenue * 100
  day = us // 86_400_000_000
  days, inv = torch.unique(day, return_inverse=True)
  per_day = torch.zeros(len(days), dtype=torch.int64, device=day.device).index_add_(0, inv, cents)

ZDW stores these cells as dictionary strings, so each conversion parses every distinct string once
(zdwb_parse_numbers) and then gathers by the codes.  The way back, from_datetime / from_decimal, formats the distinct
values once (zdwb_format_numbers) into a dense, bytewise sorted dictionary: a column valid wherever a read_table text
column is (write_table, the predicates, zdwb_merge_codes).
"""
from __future__ import annotations

from .capi import NUM_DATETIME, NUM_DECIMAL, Context
from .predicates import _text_column
from .reader import ColumnTable, FileHeader


def _parse(header: FileHeader, table: ColumnTable, k: int, kind: int, digits: int):
    codes, dct, eo, null = _text_column(header, table, k)
    with Context(codes.device.index) as ctx:
        values, ok = ctx.parse_numbers(dct, eo, kind, digits=digits, null_text=null)
    return values[codes], ok[codes]  # code -1 takes the last element, the null text's


def to_datetime(header: FileHeader, table: ColumnTable, k: int):
    """Row k of table.values (any text-like column) read as "YYYY-MM-DD HH:MM:SS[.ffffff]" or "YYYY-MM-DD": (us, valid)
    CUDA tensors with one element per row, us int64 microseconds since 1970-01-01 00:00:00 (no time zone), valid bool.
    A cell whose text is not such a date and time, or names one that does not exist (MySQL's zero date
    0000-00-00 00:00:00, 24:00:00, 1900-02-29), is 0 and not valid; so is an empty cell (code -1)."""
    return _parse(header, table, k, NUM_DATETIME, 0)


def to_decimal(header: FileHeader, table: ColumnTable, k: int, *, scale: int):
    """Row k of table.values (any text-like column) read as a decimal number times 10^scale (0..18): (v, valid) CUDA
    tensors with one element per row, v int64, valid bool.  The text is [+-]?(D+(.D*)?|.D+); a cell that is not, that has
    non-zero digits past the scale-th fraction digit, or whose value leaves int64, is 0 and not valid.  An empty cell
    (code -1) of a DECIMAL column is 0 and valid (the decoder prints it as 0.000000000000); of any other column it is not
    valid.  Scale 0 reads the integers a VARCHAR column holds."""
    return _parse(header, table, k, NUM_DECIMAL, scale)


def _format(values, valid, kind: int, digits: int):
    import torch
    if not isinstance(values, torch.Tensor) or not values.is_cuda or values.dtype != torch.int64 or values.dim() != 1:
        raise ValueError("values must be a 1-D int64 CUDA tensor")
    if valid is None:
        uniq, inv = torch.unique(values, return_inverse=True)
    else:
        if not isinstance(valid, torch.Tensor) or valid.dtype != torch.bool or valid.shape != values.shape \
                or valid.device != values.device:
            raise ValueError("valid must be a bool tensor of the shape and device of values")
        uniq, inv = torch.unique(values[valid], return_inverse=True)
    torch.cuda.current_stream(values.device).synchronize()  # the library's stream does not wait for torch's
    with Context(values.device.index) as ctx:
        m = ctx.format_numbers(uniq.contiguous(), kind, digits=digits)
    if valid is None:
        codes = m.codes[inv]
    else:
        codes = torch.full_like(values, -1)
        codes[valid] = m.codes[inv]
    return codes, (m.dict, m.entry_off)


def from_datetime(us, valid=None, *, frac_digits: int = 0):
    """int64 microseconds since 1970-01-01 (a 1-D CUDA tensor) as a DATETIME text column: (codes, (dict, entry_off)),
    ready to be a row of a ColumnTable and its entry of `dicts`.  Texts are "YYYY-MM-DD HH:MM:SS", plus '.' and
    frac_digits (0..6) digits when frac_digits > 0; every value must lie in 0001-01-01 .. 9999-12-31 23:59:59.999999 and
    be a multiple of 10^(6 - frac_digits) microseconds (ZdwError otherwise).  Rows where `valid` (a bool tensor) is False
    get code -1, an empty cell."""
    return _format(us, valid, NUM_DATETIME, frac_digits)


def from_decimal(v, valid=None, *, scale: int):
    """int64 numbers times 10^scale (a 1-D CUDA tensor) as a DECIMAL text column: (codes, (dict, entry_off)), ready to
    be a row of a ColumnTable and its entry of `dicts`.  Texts are an optional '-', the integer digits and, when
    scale > 0, '.' and exactly `scale` digits.  Rows where `valid` (a bool tensor) is False get code -1.  ZDW has no
    empty DECIMAL distinct from zero: the decoder prints such a cell as 0.000000000000, so it reads back as 0 and valid
    (to_decimal) once the table is written."""
    return _format(v, valid, NUM_DECIMAL, scale)
