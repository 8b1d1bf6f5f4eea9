"""ctypes binding of the libzdw_b200 C ABI (include/zdw_b200.h).

Fails loudly (ImportError / ZdwError) when the CUDA library is missing or no GPU is present:
there is deliberately no CPU path in the product.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from pathlib import Path

_HERE = Path(__file__).resolve().parent

STATUS_NAMES = {0: "OK", 1: "ERR_CUDA", 2: "ERR_OOM", 3: "ERR_WRONG_COLUMNS", 4: "ERR_BAD_ARG", 5: "ERR_UNSUPPORTED",
                6: "ERR_CORRUPT", 7: "ERR_TRUNCATED", 8: "ERR_ROW_COUNT", 9: "ERR_NO_DEVICE"}

EXPORTED_SYMBOLS = [
    "zdwb_abi_version", "zdwb_device_count", "zdwb_ctx_create", "zdwb_ctx_destroy", "zdwb_last_error", "zdwb_ctx_set_stream",
    "zdwb_ctx_set_tuning", "zdwb_ctx_kernel_launches", "zdwb_ctx_kernel_times", "zdwb_encode_block", "zdwb_decode_block", "zdwb_host_alloc",
    "zdwb_host_free", "zdwb_fd_to_device", "zdwb_device_to_fd", "zdwb_decode_columns", "zdwb_merge_codes",
    "zdwb_render_columns", "zdwb_match_like", "zdwb_find_strings", "zdwb_parse_numbers", "zdwb_format_numbers",
]

# zdwb_number_opts.kind
NUM_DATETIME, NUM_DECIMAL = 0, 1


class ZdwError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{STATUS_NAMES.get(code, code)}: {msg}")
        self.code = code
        self.msg = msg


def lib_path() -> Path:
    # ZDWB_LIB: developer override used by tools/ to A/B two builds of the same library (never a fallback)
    override = os.environ.get("ZDWB_LIB")
    return Path(override) if override else _HERE / "libzdw_b200.so"


class _Schema(C.Structure):
    _fields_ = [("ncols", C.c_uint32), ("types", C.POINTER(C.c_uint8))]


class _EncOpts(C.Structure):
    _fields_ = [("trim", C.c_int32), ("input_on_device", C.c_int32), ("output_on_device", C.c_int32),
                ("more_input_follows", C.c_int32), ("prev_longest_line", C.c_uint32), ("spill_cols", C.c_uint32),
                ("max_rows", C.c_uint64), ("heap_blocks", C.c_uint32), ("reserved_e", C.c_uint32)]


class _BlockOut(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("len", C.c_size_t), ("nrows", C.c_uint32), ("longest_line", C.c_uint32),
                ("tsv_consumed", C.c_uint64), ("rows_in_buffer", C.c_uint64), ("bad_row", C.c_uint32),
                ("ncols_used", C.c_uint32), ("dict_entries", C.c_uint64), ("dict_bytes", C.c_uint64),
                ("dict_index_size", C.c_uint32), ("reserved", C.c_uint32)]


class _Fill(C.Structure):
    _fields_ = [("pos", C.c_uint32), ("len", C.c_uint32), ("text", C.c_char_p)]


class _DecOpts(C.Structure):
    _fields_ = [("input_on_device", C.c_int32), ("output_on_device", C.c_int32), ("want_row_offsets", C.c_int32),
                ("at_end_of_file", C.c_int32), ("separator", C.c_uint8), ("reserved", C.c_uint8 * 7),
                ("out_col", C.POINTER(C.c_int32)), ("n_out", C.c_uint32), ("n_fills", C.c_uint32),
                ("fills", C.POINTER(_Fill)), ("rownum_pos", C.c_int32), ("validate_only", C.c_int32),
                ("first_row_number", C.c_uint64), ("want_flag_counts", C.c_int32), ("skim_only", C.c_int32)]


class _RowsOut(C.Structure):
    _fields_ = [("tsv", C.c_void_p), ("len", C.c_size_t), ("row_off", C.c_void_p), ("nrows", C.c_uint32),
                ("line_length", C.c_uint32), ("is_last", C.c_uint8), ("reserved", C.c_uint8 * 7),
                ("consumed", C.c_uint64), ("dict_bytes", C.c_uint64), ("ncols_used", C.c_uint32),
                ("reserved2", C.c_uint32), ("flag_counts", C.c_void_p)]


class _ColOpts(C.Structure):
    _fields_ = [("input_on_device", C.c_int32), ("at_end_of_file", C.c_int32), ("cols", C.POINTER(C.c_uint32)),
                ("n_cols", C.c_uint32), ("reserved", C.c_uint32)]


class _ColsOut(C.Structure):
    _fields_ = [("values", C.c_void_p), ("dict", C.c_void_p), ("entry_off", C.c_void_p), ("dict_entries", C.c_uint64),
                ("dict_bytes", C.c_uint64), ("consumed", C.c_uint64), ("nrows", C.c_uint32), ("line_length", C.c_uint32),
                ("is_last", C.c_uint8), ("reserved", C.c_uint8 * 3), ("ncols_used", C.c_uint32)]


class _CodePart(C.Structure):
    _fields_ = [("dict", C.c_void_p), ("entry_off", C.c_void_p), ("entries", C.c_uint64), ("dict_bytes", C.c_uint64),
                ("codes", C.c_void_p), ("n", C.c_uint64)]


class _MergeOut(C.Structure):
    _fields_ = [("codes", C.c_void_p), ("dict", C.c_void_p), ("entry_off", C.c_void_p), ("entries", C.c_uint64),
                ("dict_bytes", C.c_uint64), ("n", C.c_uint64)]


class _RenderOut(C.Structure):
    _fields_ = [("tsv", C.c_void_p), ("len", C.c_uint64)]


class _LikeOpts(C.Structure):
    _fields_ = [("pattern", C.c_char_p), ("pattern_len", C.c_uint64), ("null_text", C.c_char_p), ("null_text_len", C.c_uint64),
                ("escape", C.c_int32), ("ignore_case", C.c_int32)]


class _MatchOut(C.Structure):
    _fields_ = [("flags", C.c_void_p), ("n", C.c_uint64)]


class _Strings(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("bytes_len", C.c_uint64), ("off", C.c_void_p), ("n", C.c_uint64)]


class _FindOut(C.Structure):
    _fields_ = [("rank", C.c_void_p), ("found", C.c_void_p), ("n", C.c_uint64)]


class _NumberOpts(C.Structure):
    _fields_ = [("kind", C.c_int32), ("digits", C.c_int32), ("null_text", C.c_char_p), ("null_text_len", C.c_uint64)]


class _ParseOut(C.Structure):
    _fields_ = [("values", C.c_void_p), ("ok", C.c_void_p), ("n", C.c_uint64)]


_lib = None


def _copy_out(ptr: int, n: int) -> bytes:
    """n bytes at a raw host pointer (ctypes.string_at takes a C int: it fails beyond 2 GiB)."""
    if not n:
        return b""
    return bytes((C.c_uint8 * n).from_address(ptr))


def load_library():
    """Loads libzdw_b200.so; raises ImportError if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not p.exists():
        raise ImportError(f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(zdw_b200 has no CPU fallback)")
    L = C.CDLL(str(p))
    L.zdwb_abi_version.restype = C.c_int
    L.zdwb_device_count.restype = C.c_int
    L.zdwb_ctx_create.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_void_p)]
    L.zdwb_ctx_destroy.argtypes = [C.c_void_p]
    L.zdwb_ctx_destroy.restype = None
    L.zdwb_last_error.argtypes = [C.c_void_p]
    L.zdwb_last_error.restype = C.c_char_p
    L.zdwb_ctx_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    L.zdwb_ctx_set_tuning.argtypes = [C.c_void_p, C.c_char_p, C.c_longlong]
    L.zdwb_ctx_kernel_launches.argtypes = [C.c_void_p]
    L.zdwb_ctx_kernel_launches.restype = C.c_ulonglong
    L.zdwb_ctx_kernel_times.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
    L.zdwb_ctx_kernel_times.restype = C.c_size_t
    L.zdwb_encode_block.argtypes = [C.c_void_p, C.POINTER(_Schema), C.c_void_p, C.c_size_t, C.POINTER(_EncOpts),
                                    C.POINTER(_BlockOut)]
    L.zdwb_decode_block.argtypes = [C.c_void_p, C.POINTER(_Schema), C.c_void_p, C.c_size_t, C.POINTER(_DecOpts),
                                    C.POINTER(_RowsOut)]
    L.zdwb_decode_columns.argtypes = [C.c_void_p, C.POINTER(_Schema), C.c_void_p, C.c_size_t, C.POINTER(_ColOpts),
                                      C.POINTER(_ColsOut)]
    L.zdwb_merge_codes.argtypes = [C.c_void_p, C.POINTER(_CodePart), C.c_uint32, C.POINTER(_MergeOut)]
    L.zdwb_render_columns.argtypes = [C.c_void_p, C.POINTER(_Schema), C.POINTER(_CodePart), C.POINTER(_RenderOut)]
    L.zdwb_match_like.argtypes = [C.c_void_p, C.POINTER(_CodePart), C.POINTER(_LikeOpts), C.POINTER(_MatchOut)]
    L.zdwb_find_strings.argtypes = [C.c_void_p, C.POINTER(_CodePart), C.POINTER(_Strings), C.POINTER(_FindOut)]
    L.zdwb_parse_numbers.argtypes = [C.c_void_p, C.POINTER(_CodePart), C.POINTER(_NumberOpts), C.POINTER(_ParseOut)]
    L.zdwb_format_numbers.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(_NumberOpts), C.POINTER(_MergeOut)]
    L.zdwb_host_alloc.argtypes = [C.c_size_t]
    L.zdwb_host_alloc.restype = C.c_void_p
    L.zdwb_host_free.argtypes = [C.c_void_p]
    L.zdwb_host_free.restype = None
    L.zdwb_fd_to_device.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_size_t, C.POINTER(C.c_void_p)]
    L.zdwb_device_to_fd.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_longlong]
    _lib = L
    return L


@dataclass
class EncodedBlock:
    data: bytes | None      # block bytes (None when left on the device)
    dev_ptr: int            # device pointer when output_on_device
    length: int
    nrows: int
    longest_line: int
    tsv_consumed: int
    rows_in_buffer: int
    ncols_used: int
    dict_entries: int
    dict_bytes: int
    dict_index_size: int


@dataclass
class DecodedBlock:
    tsv: bytes | None
    dev_ptr: int
    length: int
    row_off: list | None
    nrows: int
    line_length: int
    is_last: bool
    consumed: int
    dict_bytes: int
    ncols_used: int
    flag_counts: list | None = None


# column types whose cells zdwb_decode_columns gives as dictionary codes (include/zdw_b200.h): VARCHAR, TEXT, DATETIME,
# CHAR_2, DECIMAL, TINYTEXT, MEDIUMTEXT, LONGTEXT (the library's is_text_like, csrc/common.cuh)
TEXT_LIKE_TYPES = frozenset({0, 1, 2, 3, 11, 16, 17, 18})


@dataclass
class ColumnBlock:
    """One block decoded into typed device columns (zdwb_decode_columns): row k of `values` is the k-th requested column.

    values     (K, nrows) int64 CUDA tensor.  Text-like columns hold codes into this block's dictionary (-1 = no value: the
               empty string, "0.000000000000" for DECIMAL); unsigned integers hold their bits (`.view(torch.uint64)`),
               signed integers their value, CHAR columns the stored tuple (low byte = the character).
    dict       uint8 CUDA tensor: the block's dictionary, origin NUL byte included (empty when no text column was asked for).
    entry_off  int64 CUDA tensor of dict_entries + 1 offsets: entry i is dict[entry_off[i] : entry_off[i + 1] - 1].
    The entries are sorted bytewise, so within a block codes compare like the strings.
    """
    values: object
    dict: object
    entry_off: object
    columns: list            # file column index of every row of `values`
    nrows: int
    consumed: int            # bytes the block occupied: the next block starts there
    is_last: bool
    line_length: int
    ncols_used: int

    def strings(self, k: int) -> list:
        """The texts of row k of `values` (a text-like column) on the host: bytes per row, None for code -1."""
        return _strings(self.values[k], self.dict, self.entry_off)


def _strings(codes, dct, entry_off) -> list:
    """Host texts of a 1-D code tensor into (dict, entry_off): bytes per code, None for -1."""
    d = bytes(dct.cpu().numpy().tobytes()) if dct.numel() else b""
    eo = entry_off.cpu().tolist()
    return [None if c < 0 else d[eo[c]:eo[c + 1] - 1] for c in codes.cpu().tolist()]


@dataclass
class MergedCodes:
    """The result of Context.merge_codes (zdwb_merge_codes).

    codes      int64 CUDA tensor: the parts' codes, concatenated in order, into `dict` (-1 stays -1).
    dict       uint8 CUDA tensor: origin NUL byte, then every entry NUL-terminated (empty when no code references one).
    entry_off  int64 CUDA tensor of entries + 1 offsets: entry i is dict[entry_off[i] : entry_off[i + 1] - 1].
    The entries are distinct, sorted bytewise, and each is referenced by a code: codes 0 .. entries - 1 all occur, they
    compare like their strings, and two codes are equal iff their strings are.
    """
    codes: object
    dict: object
    entry_off: object

    @property
    def entries(self) -> int:
        return self.entry_off.numel() - 1

    def strings(self) -> list:
        """The texts of `codes` on the host: bytes per code, None for -1."""
        return _strings(self.codes, self.dict, self.entry_off)


class _DeviceArray:
    """A device range seen through __cuda_array_interface__ (so that torch can copy it)."""

    def __init__(self, ptr: int, shape: tuple, typestr: str):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 3,
                                         "strides": None, "stream": None}


def _device_tensors(torch, device: int, copy_stream, ranges):
    """Tensors of their own with the contents of context-owned device ranges [(ptr, shape, typestr, dtype), ...].

    The context re-uses its memory at its next call, so the copies must be complete before this returns.  They run on
    `copy_stream`, which holds nothing else, and the host waits for them there: work the caller has queued on torch's
    current stream neither delays them nor runs after them.  The tensors are handed to the current stream afterwards
    (record_stream), so that the caching allocator does not give their memory to the copy stream while work on the
    current stream may still read them."""
    cur = torch.cuda.current_stream(device)
    out = []
    with torch.cuda.stream(copy_stream):
        for ptr, shape, typestr, dtype in ranges:
            if not ptr or any(n == 0 for n in shape):
                out.append(torch.empty(shape, dtype=dtype, device=f"cuda:{device}"))
            else:
                out.append(torch.as_tensor(_DeviceArray(ptr, shape, typestr), device=f"cuda:{device}").clone())
    copy_stream.synchronize()
    for t in out:
        t.record_stream(cur)
    return out


class Context:
    """One GPU context (zdwb_ctx).  Not thread-safe; one per host thread / GPU."""

    def __init__(self, device: int = 0, workspace_hint: int = 0):
        self._L = load_library()
        h = C.c_void_p()
        rc = self._L.zdwb_ctx_create(device, workspace_hint, C.byref(h))
        if rc != 0:
            raise ZdwError(rc, "zdwb_ctx_create failed (is a CUDA device visible? zdw_b200 has no CPU fallback)")
        self._h = h
        self.device = device
        self._copy_stream = None  # torch stream of the decode_columns copies (created at the first call)

    def close(self):
        if getattr(self, "_h", None):
            self._L.zdwb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def last_error(self) -> str:
        return self._L.zdwb_last_error(self._h).decode("latin1")

    def set_stream(self, cuda_stream: int | None):
        rc = self._L.zdwb_ctx_set_stream(self._h, C.c_void_p(cuda_stream or 0))
        if rc:
            raise ZdwError(rc, self.last_error())

    def set_tuning(self, name: str, value: int):
        rc = self._L.zdwb_ctx_set_tuning(self._h, name.encode(), value)
        if rc:
            raise ZdwError(rc, f"unknown tuning knob {name}")

    def kernel_launches(self) -> int:
        return int(self._L.zdwb_ctx_kernel_launches(self._h))

    def kernel_times(self) -> dict:
        """{kernel name: (launches, total_ms)} since the last call (needs set_tuning("kernel_timing", 1))."""
        buf = C.create_string_buffer(1 << 16)
        self._L.zdwb_ctx_kernel_times(self._h, buf, len(buf))
        out = {}
        for line in buf.value.decode().splitlines():
            name, cnt, ms = line.split("\t")
            out[name] = (int(cnt), float(ms))
        return out

    # ------------------------------------------------------------------ file descriptor <-> device
    def fd_to_device(self, fd: int, offset: int, n: int) -> int:
        """`n` bytes of fd from `offset` (< 0: read() at its position) to a device buffer of the context; returns its address."""
        dev = C.c_void_p()
        rc = self._L.zdwb_fd_to_device(self._h, fd, offset, n, C.byref(dev))
        if rc:
            raise ZdwError(rc, self.last_error())
        return int(dev.value or 0)

    def device_to_fd(self, dev_ptr: int, n: int, fd: int, offset: int):
        """`n` device bytes to fd at `offset` (< 0: write() at its position)."""
        rc = self._L.zdwb_device_to_fd(self._h, C.c_void_p(dev_ptr), n, fd, offset)
        if rc:
            raise ZdwError(rc, self.last_error())

    # ------------------------------------------------------------------ encode
    def encode_block(self, types, tsv, n: int | None = None, *, trim=False, input_on_device=False,
                     output_on_device=False, prev_longest_line=0, max_rows=0, more_input_follows=False,
                     spill_cols=0, heap_blocks=0) -> EncodedBlock:
        """tsv: bytes-like (host) or an int device pointer (input_on_device=True, n required)."""
        tarr = (C.c_uint8 * max(len(types), 1))(*types)
        sch = _Schema(len(types), C.cast(tarr, C.POINTER(C.c_uint8)))
        if input_on_device:
            ptr = C.c_void_p(int(tsv))
            assert n is not None
        else:
            keep = tsv if isinstance(tsv, (bytes, bytearray)) else bytes(tsv)
            n = len(keep) if n is None else n
            ptr = C.cast(C.c_char_p(bytes(keep)), C.c_void_p) if not isinstance(keep, bytes) else C.cast(C.c_char_p(keep), C.c_void_p)
        o = _EncOpts(int(trim), int(input_on_device), int(output_on_device), int(more_input_follows), prev_longest_line,
                     int(spill_cols), max_rows, int(heap_blocks), 0)
        out = _BlockOut()
        rc = self._L.zdwb_encode_block(self._h, C.byref(sch), ptr, n, C.byref(o), C.byref(out))
        if rc:
            e = ZdwError(rc, self.last_error())
            e.bad_row = out.bad_row
            raise e
        data = None
        if not output_on_device:
            data = _copy_out(out.bytes, out.len)
        return EncodedBlock(data, int(out.bytes or 0), out.len, out.nrows, out.longest_line, out.tsv_consumed,
                            out.rows_in_buffer, out.ncols_used, out.dict_entries, out.dict_bytes, out.dict_index_size)

    # ------------------------------------------------------------------ decode
    def decode_block(self, types, zdw, avail: int | None = None, *, input_on_device=False, output_on_device=False,
                     want_row_offsets=False, at_end_of_file=True, separator=b"\t", out_col=None, n_out=0, fills=None,
                     rownum_pos=-1, first_row_number=1, validate_only=False, want_flag_counts=False,
                     skim_only=False) -> DecodedBlock:
        """fills: {output position: bytes} constant texts for positions no file column maps to."""
        tarr = (C.c_uint8 * max(len(types), 1))(*types)
        sch = _Schema(len(types), C.cast(tarr, C.POINTER(C.c_uint8)))
        if input_on_device:
            ptr = C.c_void_p(int(zdw))
            assert avail is not None
        else:
            keep = bytes(zdw)
            avail = len(keep) if avail is None else avail
            ptr = C.cast(C.c_char_p(keep), C.c_void_p)
        oc = None
        if out_col is not None:
            oc = (C.c_int32 * len(out_col))(*out_col)
        fl = None
        if fills:
            fl = (_Fill * len(fills))(*[_Fill(int(k), len(v), v) for k, v in fills.items()])
        o = _DecOpts(int(input_on_device), int(output_on_device), int(want_row_offsets), int(at_end_of_file),
                     separator[0], (C.c_uint8 * 7)(), C.cast(oc, C.POINTER(C.c_int32)) if oc is not None else None,
                     n_out, len(fills) if fills else 0, C.cast(fl, C.POINTER(_Fill)) if fl is not None else None,
                     rownum_pos, int(validate_only), first_row_number, int(want_flag_counts), int(skim_only))
        out = _RowsOut()
        rc = self._L.zdwb_decode_block(self._h, C.byref(sch), ptr, avail, C.byref(o), C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        tsv = None
        offs = None
        if not output_on_device:
            tsv = _copy_out(out.tsv, out.len)
            if want_row_offsets and out.row_off:
                arr = (C.c_uint64 * (out.nrows + 1)).from_address(out.row_off)
                offs = list(arr)
        counts = None
        if want_flag_counts and out.flag_counts:
            counts = list((C.c_uint64 * out.ncols_used).from_address(out.flag_counts))
        return DecodedBlock(tsv, int(out.tsv or 0), out.len, offs, out.nrows, out.line_length, bool(out.is_last),
                            out.consumed, out.dict_bytes, out.ncols_used, counts)

    # ------------------------------------------------------------------ columnar decode
    def decode_columns(self, types, zdw, columns, avail: int | None = None, *, input_on_device=False, at_end_of_file=True,
                       offset: int = 0) -> ColumnBlock:
        """Decodes the block at zdw[offset:] into typed device columns (see ColumnBlock).  columns: file column indices,
        in the order of the output rows.  zdw: bytes-like (host) or an int device pointer (input_on_device=True, avail
        required).  The tensors are copies, complete when this returns: they stay valid after the next call on the context,
        whatever is queued on torch's current stream."""
        import torch  # (only needed here: the rest of the binding works without it)

        tarr = (C.c_uint8 * max(len(types), 1))(*types)
        sch = _Schema(len(types), C.cast(tarr, C.POINTER(C.c_uint8)))
        if input_on_device:
            if avail is None:
                raise ValueError("decode_columns: `avail` is required with input_on_device")
            ptr = C.c_void_p(int(zdw) + offset)
        else:
            keep = zdw if isinstance(zdw, bytes) else bytes(zdw)
            avail = len(keep) - offset if avail is None else avail
            ptr = C.c_void_p(C.cast(C.c_char_p(keep), C.c_void_p).value + offset)
        cols = [int(c) for c in columns]
        carr = (C.c_uint32 * max(len(cols), 1))(*cols)
        o = _ColOpts(int(input_on_device), int(at_end_of_file), C.cast(carr, C.POINTER(C.c_uint32)), len(cols), 0)
        out = _ColsOut()
        rc = self._L.zdwb_decode_columns(self._h, C.byref(sch), ptr, avail, C.byref(o), C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        dev = self.device
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        values, dct, eo = _device_tensors(torch, dev, self._copy_stream, [
            (out.values or 0, (len(cols), out.nrows), "<i8", torch.int64),
            (out.dict or 0, (out.dict_bytes if out.dict else 0,), "|u1", torch.uint8),
            (out.entry_off or 0, (out.dict_entries + 1 if out.entry_off else 0,), "<i8", torch.int64)])
        return ColumnBlock(values, dct, eo, cols, out.nrows, out.consumed, bool(out.is_last), out.line_length, out.ncols_used)

    # ------------------------------------------------------------------ merged dictionaries
    def merge_codes(self, parts) -> MergedCodes:
        """One sorted dictionary for codes into many (zdwb_merge_codes; see MergedCodes).  parts: a sequence of
        (dict, entry_off, codes) CUDA tensors on the context's device, e.g. (blk.dict, blk.entry_off, blk.values[k]) of
        ColumnBlocks; codes 1-D contiguous int64, entry_off int64 (or uint64) with entries + 1 offsets.  The tensors
        must hold their final contents when the call is made (those of decode_columns do): the context's stream does not
        wait for torch's.  The results are copies, complete when this returns, as with decode_columns."""
        import torch

        dev = self.device
        arr = (_CodePart * max(len(parts), 1))()
        for i, (dct, eo, codes) in enumerate(parts):
            for name, t in (("dict", dct), ("entry_off", eo), ("codes", codes)):
                if not t.is_cuda or t.device.index != dev or not t.is_contiguous():
                    raise ValueError(f"merge_codes: part {i}: {name} must be a contiguous tensor on cuda:{dev}")
            if codes.dtype != torch.int64 or codes.dim() != 1:
                raise ValueError(f"merge_codes: part {i}: codes must be a 1-D int64 tensor")
            if eo.dtype not in (torch.int64, torch.uint64) or dct.dtype != torch.uint8:
                raise ValueError(f"merge_codes: part {i}: dict must be uint8 and entry_off int64")
            entries = max(eo.numel() - 1, 0)
            arr[i] = _CodePart(dct.data_ptr() if dct.numel() else None, eo.data_ptr() if eo.numel() else None, entries,
                               dct.numel(), codes.data_ptr() if codes.numel() else None, codes.numel())
        out = _MergeOut()
        rc = self._L.zdwb_merge_codes(self._h, arr, len(parts), C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        codes, dct, eo = _device_tensors(torch, dev, self._copy_stream, [
            (out.codes or 0, (out.n,), "<i8", torch.int64),
            (out.dict or 0, (out.dict_bytes,), "|u1", torch.uint8),
            (out.entry_off or 0, (out.entries + 1,), "<i8", torch.int64)])
        return MergedCodes(codes, dct, eo)

    # ------------------------------------------------------------------ columns back to rows
    def render_columns(self, types, cells, dicts) -> tuple[int, int]:
        """TSV rows of typed device columns (zdwb_render_columns; include/zdw_b200.h gives the text of every cell), which
        encode_block(types, ptr, length, input_on_device=True) encodes back into the same cells.  types: the column
        types; cells: a sequence of 1-D int64 CUDA tensors, or a 2-D one (row k = column k), on the context's device;
        dicts: per column (dict, entry_off) for a text-like column (as ColumnTable.dicts holds them), None for the
        others.  The tensors must hold their final contents when the call is made, as with merge_codes.  Returns
        (device pointer, length) of the rows: a buffer of the context, valid until its next render_columns call."""
        import torch

        dev = self.device
        if isinstance(cells, torch.Tensor) and cells.dim() == 2:
            cells = list(cells)
        if len(cells) != len(types) or len(dicts) != len(types):
            raise ValueError(f"render_columns: {len(types)} types, {len(cells)} columns of cells and {len(dicts)} dicts")
        arr = (_CodePart * max(len(types), 1))()
        for k, (codes, dd) in enumerate(zip(cells, dicts)):
            if not isinstance(codes, torch.Tensor) or not codes.is_cuda or codes.device.index != dev:
                raise ValueError(f"render_columns: column {k}: cells must be a tensor on cuda:{dev}")
            if codes.dtype != torch.int64 or codes.dim() != 1 or not codes.is_contiguous():
                raise ValueError(f"render_columns: column {k}: cells must be a contiguous 1-D int64 tensor")
            dptr = eptr = None
            entries = nbytes = 0
            if dd is not None:
                dct, eo = dd
                for name, t in (("dict", dct), ("entry_off", eo)):
                    if not t.is_cuda or t.device.index != dev or not t.is_contiguous():
                        raise ValueError(f"render_columns: column {k}: {name} must be a contiguous tensor on cuda:{dev}")
                if eo.dtype not in (torch.int64, torch.uint64) or dct.dtype != torch.uint8:
                    raise ValueError(f"render_columns: column {k}: dict must be uint8 and entry_off int64")
                entries = max(eo.numel() - 1, 0)
                nbytes = dct.numel()
                dptr = dct.data_ptr() if nbytes else None
                eptr = eo.data_ptr() if eo.numel() else None
            arr[k] = _CodePart(dptr, eptr, entries, nbytes, codes.data_ptr() if codes.numel() else None, codes.numel())
        tarr = (C.c_uint8 * max(len(types), 1))(*types)
        sch = _Schema(len(types), C.cast(tarr, C.POINTER(C.c_uint8)))
        out = _RenderOut()
        rc = self._L.zdwb_render_columns(self._h, C.byref(sch), arr, C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        return int(out.tsv or 0), int(out.len)

    # ------------------------------------------------------------------ predicates over a dictionary
    def _dict_part(self, who: str, dct, eo) -> _CodePart:
        import torch
        for name, t in (("dict", dct), ("entry_off", eo)):
            if not isinstance(t, torch.Tensor) or not t.is_cuda or t.device.index != self.device or not t.is_contiguous():
                raise ValueError(f"{who}: {name} must be a contiguous tensor on cuda:{self.device}")
        if eo.dtype not in (torch.int64, torch.uint64) or dct.dtype != torch.uint8:
            raise ValueError(f"{who}: dict must be uint8 and entry_off int64")
        return _CodePart(dct.data_ptr() if dct.numel() else None, eo.data_ptr() if eo.numel() else None,
                         max(eo.numel() - 1, 0), dct.numel(), None, 0)

    def match_like(self, dct, entry_off, pattern: bytes, *, escape: bytes | None = b"\\", ignore_case=False,
                   null_text: bytes = b""):
        """SQL LIKE of every entry of a dictionary (zdwb_match_like; include/zdw_b200.h gives the rules): a bool CUDA
        tensor of entries + 1 flags, the last one for `null_text`, the text of code -1.  So `flags[codes]` is the answer
        per cell, code -1 included.  dct, entry_off: a dictionary as ColumnTable.dicts[k] or ColumnBlock.dict /
        entry_off hold it, on the context's device, with their final contents (as with merge_codes).  escape: one byte,
        or None for none.  The result is a copy, complete when this returns."""
        import torch
        part = self._dict_part("match_like", dct, entry_off)
        if escape is not None and len(escape) != 1:
            raise ValueError("match_like: escape must be one byte or None")
        pattern, null_text = bytes(pattern), bytes(null_text)
        o = _LikeOpts(pattern, len(pattern), null_text, len(null_text), -1 if escape is None else escape[0], int(bool(ignore_case)))
        out = _MatchOut()
        rc = self._L.zdwb_match_like(self._h, C.byref(part), C.byref(o), C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        (flags,) = _device_tensors(torch, self.device, self._copy_stream, [(out.flags or 0, (out.n,), "|u1", torch.uint8)])
        return flags.view(torch.bool)

    def find_strings(self, dct, entry_off, strings):
        """lower_bound of every string of `strings` (a sequence of bytes) among the entries of a sorted dictionary
        (zdwb_find_strings): (rank, found) CUDA tensors, rank int64 = the number of entries bytewise less than the string,
        found bool = entry rank equals it.  The dictionary is taken as by match_like; the strings go to the device in one
        buffer.  The results are copies, complete when this returns."""
        import torch
        dev = self.device
        part = self._dict_part("find_strings", dct, entry_off)
        import numpy as np
        strings = [s if isinstance(s, bytes) else bytes(s) for s in strings]
        offs = np.zeros(len(strings) + 1, dtype=np.int64)
        np.cumsum(np.fromiter(map(len, strings), dtype=np.int64, count=len(strings)), out=offs[1:])
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        # the queries are uploaded on the copy stream and complete before the call: torch's current stream may be busy
        with torch.cuda.stream(self._copy_stream):
            blob = b"".join(strings)
            qb = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(f"cuda:{dev}") if blob else \
                torch.empty(0, dtype=torch.uint8, device=f"cuda:{dev}")
            qo = torch.from_numpy(offs).to(f"cuda:{dev}")
        self._copy_stream.synchronize()
        q = _Strings(qb.data_ptr() if qb.numel() else None, qb.numel(), qo.data_ptr(), len(strings))
        out = _FindOut()
        rc = self._L.zdwb_find_strings(self._h, C.byref(part), C.byref(q), C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        rank, found = _device_tensors(torch, dev, self._copy_stream, [
            (out.rank or 0, (out.n,), "<i8", torch.int64), (out.found or 0, (out.n,), "|u1", torch.uint8)])
        return rank, found.view(torch.bool)

    # ------------------------------------------------------------------ numbers from and to text
    def parse_numbers(self, dct, entry_off, kind: int, *, digits: int = 0, null_text: bytes = b""):
        """The number of every entry of a dictionary (zdwb_parse_numbers; include/zdw_b200.h gives the grammars): kind
        NUM_DATETIME gives microseconds since 1970-01-01, NUM_DECIMAL the number times 10^digits.  Returns (values, ok)
        CUDA tensors of entries + 1 elements, int64 and bool, the last one for `null_text`, the text of code -1; ok is
        False (and the value 0) where the text is not in the grammar or its number does not fit.  So `values[codes]` is
        the answer per cell, code -1 included.  The dictionary is taken as by match_like.  The results are copies,
        complete when this returns."""
        import torch
        part = self._dict_part("parse_numbers", dct, entry_off)
        null_text = bytes(null_text)
        o = _NumberOpts(int(kind), int(digits), null_text, len(null_text))
        out = _ParseOut()
        rc = self._L.zdwb_parse_numbers(self._h, C.byref(part), C.byref(o), C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        values, ok = _device_tensors(torch, self.device, self._copy_stream, [
            (out.values or 0, (out.n,), "<i8", torch.int64), (out.ok or 0, (out.n,), "|u1", torch.uint8)])
        return values, ok.view(torch.bool)

    def format_numbers(self, values, kind: int, *, digits: int = 0) -> MergedCodes:
        """Strictly increasing numbers (a 1-D int64 CUDA tensor on the context's device, e.g. torch.unique's output, with
        its final contents) as a dictionary (zdwb_format_numbers): kind NUM_DATETIME writes microseconds since 1970-01-01
        as "YYYY-MM-DD HH:MM:SS" plus `digits` (0..6) fraction digits, NUM_DECIMAL writes v / 10^digits (0..18) with
        exactly `digits` fraction digits.  Returns MergedCodes: codes[i] is the code of values[i]'s text in the dense,
        bytewise sorted dictionary.  The results are copies, complete when this returns."""
        import torch
        dev = self.device
        if not isinstance(values, torch.Tensor) or not values.is_cuda or values.device.index != dev:
            raise ValueError(f"format_numbers: values must be a tensor on cuda:{dev}")
        if values.dtype != torch.int64 or values.dim() != 1 or not values.is_contiguous():
            raise ValueError("format_numbers: values must be a contiguous 1-D int64 tensor")
        o = _NumberOpts(int(kind), int(digits), None, 0)
        out = _MergeOut()
        rc = self._L.zdwb_format_numbers(self._h, C.c_void_p(values.data_ptr() if values.numel() else None), values.numel(),
                                         C.byref(o), C.byref(out))
        if rc:
            raise ZdwError(rc, self.last_error())
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        codes, dct, eo = _device_tensors(torch, dev, self._copy_stream, [
            (out.codes or 0, (out.n,), "<i8", torch.int64),
            (out.dict or 0, (out.dict_bytes,), "|u1", torch.uint8),
            (out.entry_off or 0, (out.entries + 1,), "<i8", torch.int64)])
        return MergedCodes(codes, dct, eo)
