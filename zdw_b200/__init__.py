"""zdw_b200 -- B200 (sm_100a) implementation of the adobe/zdw hot path.

The product is native: `libzdw_b200.so` (hand-written CUDA kernels behind the C ABI declared in
include/zdw_b200.h) plus the C++ host classes/CLIs under zdw_b200/host.  This Python package holds
the ctypes binding of that ABI (capi: Context, used by the test-suite and bench.py) and a reader
that decodes ZDW files into typed CUDA tensors (reader: read_header, read_columns; one ColumnBlock
per block, decoded on the GPU by zdwb_decode_columns; read_table: one ColumnTable per file, its text
columns merged into file-wide dictionaries by zdwb_merge_codes) and a writer that goes the other way (writer:
write_table renders a ColumnTable's blocks to TSV on the GPU with zdwb_render_columns and encodes them with
zdwb_encode_block) and filters on text columns (predicates: like, isin, between, answered once per dictionary entry by
zdwb_match_like and zdwb_find_strings) and reads DATETIME and DECIMAL columns as numbers and writes numbers back
(numbers: to_datetime, to_decimal, from_datetime, from_decimal, on zdwb_parse_numbers and zdwb_format_numbers).  It
contains no compute of its own and no CPU fallback; torch is only imported by the columnar calls.
"""
from .capi import (  # noqa: F401
    ColumnBlock,
    Context,
    EncodedBlock,
    DecodedBlock,
    MergedCodes,
    ZdwError,
    lib_path,
    load_library,
)
from .reader import ColumnTable, FileHeader, read_columns, read_header, read_table  # noqa: F401
from .writer import write_table  # noqa: F401
from .predicates import between, isin, like  # noqa: F401
from .numbers import from_datetime, from_decimal, to_datetime, to_decimal  # noqa: F401

__all__ = ["Context", "EncodedBlock", "DecodedBlock", "ColumnBlock", "MergedCodes", "ZdwError", "FileHeader", "ColumnTable",
           "lib_path", "load_library", "read_columns", "read_header", "read_table",
           "write_table", "like", "isin", "between", "to_datetime", "to_decimal", "from_datetime", "from_decimal"]
