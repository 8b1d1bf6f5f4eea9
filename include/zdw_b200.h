/*
 * zdw_b200.h -- C ABI of libzdw_b200.so, the B200 (sm_100a) implementation of the adobe/zdw hot path.
 *
 * The reference (adobe/zdw, cplusplus/) has no plugin/FFI interface: its hot path sits inside two
 * C++ classes.  This ABI is the seam a maintainer cuts at: the bodies of the functions cited below
 * are replaced by one call each, everything around them (CLI, .desc.sql, file header, compressor
 * pipe, block stitching) stays host C++.  See INTEGRATION.md for the binding on the reference side.
 *
 *   zdwb_encode_block   replaces, for one ZDW block,
 *        ConvertToZDW::parseInput            ConvertToZDW.cpp:329-414   (pass 1)
 *        GetNextRow / GetDataRow             getnextrow.cpp:26-84, ConvertToZDW.cpp:265-323, :1048-1067
 *        Dictionary::insert/write/getOffset  dictionary.cpp:31-111
 *        writeLookupColumnStats              ConvertToZDW.cpp:417-483
 *        writeBlockRows                      ConvertToZDW.cpp:486-606   (pass 2)
 *        and the block header fields         ConvertToZDW.cpp:839-842
 *   zdwb_decode_block   replaces, for one ZDW block,
 *        UnconvertFromZDW_Base::parseBlockHeader   UnconvertFromZDW.cpp:758-1000
 *        UnconvertFromZDW<T>::readNextRow          UnconvertFromZDW.cpp:1270-1464 (+GetWord :359-371,
 *        llutoa/lltoa :318-356, outputDefault :1224-1266) for all rows of the block
 *   zdwb_decode_columns (no counterpart in the reference) decodes a block into typed device columns instead
 *        of text: one int64 per cell, text as codes into the block's sorted dictionary
 *   zdwb_merge_codes (no counterpart either) merges the dictionaries of many blocks into one sorted dictionary and
 *        re-codes their codes into it
 *   zdwb_render_columns (no counterpart either) renders typed device columns back to TSV rows, the input of
 *        zdwb_encode_block: the way from columns back to a ZDW file
 *   zdwb_match_like, zdwb_find_strings (no counterpart either) answer LIKE and string lookups over a sorted dictionary,
 *        once per distinct string: the filters on text columns
 *   zdwb_parse_numbers, zdwb_format_numbers (no counterpart either) read DATETIME and DECIMAL dictionary strings as
 *        numbers and write numbers back as a sorted dictionary
 *
 * Plain C types only; int status codes; no exceptions and no C++ types cross the boundary.  Outputs
 * are owned by the context and stay valid until the next call on the same context.  One context per
 * host thread / GPU.  There is no CPU fallback: every entry point fails with ZDWB_ERR_NO_DEVICE or
 * ZDWB_ERR_CUDA when the GPU path is unavailable.
 */
#ifndef ZDW_B200_H
#define ZDW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZDWB_ABI_VERSION 5

/* status codes (mapped to the reference's ERR_CODE enums by the host classes) */
enum {
  ZDWB_OK = 0,
  ZDWB_ERR_CUDA = 1,          /* CUDA runtime/driver error                     -> PROCESSING_ERROR / CONVERSION_FAILED */
  ZDWB_ERR_OOM = 2,           /* device or pinned allocation failed            -> OUT_OF_MEMORY (ConvertToZDW.h:52) */
  ZDWB_ERR_WRONG_COLUMNS = 3, /* a row's field count != schema                 -> WRONG_NUM_OF_COLUMNS_ON_A_ROW (15) */
  ZDWB_ERR_BAD_ARG = 4,       /* NULL / inconsistent arguments                 -> BAD_PARAMETER */
  ZDWB_ERR_UNSUPPORTED = 5,   /* input outside the supported envelope (see DESIGN.md limits) */
  ZDWB_ERR_CORRUPT = 6,       /* dictionary offset out of range                -> CORRUPTED_DATA_ERROR (9) */
  ZDWB_ERR_TRUNCATED = 7,     /* block runs past the bytes supplied            -> GZREAD_FAILED (2) */
  ZDWB_ERR_ROW_COUNT = 8,     /* fewer rows than the block header promises     -> ROW_COUNT_ERR (8) */
  ZDWB_ERR_NO_DEVICE = 9      /* no usable CUDA device */
};

/* column type ids as stored in the file: zdw_column_type_constants.h:17-35 */
enum {
  ZDWB_VARCHAR = 0, ZDWB_TEXT = 1, ZDWB_DATETIME = 2, ZDWB_CHAR_2 = 3, ZDWB_VISID_LOW = 4,
  ZDWB_VISID_HIGH = 5, ZDWB_CHAR = 6, ZDWB_TINY = 7, ZDWB_SHORT = 8, ZDWB_LONG = 9, ZDWB_LONGLONG = 10,
  ZDWB_DECIMAL = 11, ZDWB_TINY_SIGNED = 12, ZDWB_SHORT_SIGNED = 13, ZDWB_LONG_SIGNED = 14,
  ZDWB_LONGLONG_SIGNED = 15, ZDWB_TINYTEXT = 16, ZDWB_MEDIUMTEXT = 17, ZDWB_LONGTEXT = 18
};

typedef struct zdwb_ctx zdwb_ctx;

/* ---- context -------------------------------------------------------------------------------- */

/* Creates a context bound to CUDA device `device`.  `workspace_hint` (bytes, 0 = default) seeds the
 * device memory pool so that steady-state calls do not allocate. */
int zdwb_ctx_create(int device, size_t workspace_hint, zdwb_ctx** out);
void zdwb_ctx_destroy(zdwb_ctx* ctx);

/* Human-readable description of the last failure on this context ("" if none). */
const char* zdwb_last_error(const zdwb_ctx* ctx);

/* Run all work of this context on the given cudaStream_t (NULL = the context's own stream).  Lets a
 * harness time the kernels with events recorded on its own stream. */
int zdwb_ctx_set_stream(zdwb_ctx* ctx, void* cuda_stream);

/* Tuning / test knobs (name = value); every default is what the measurements in DESIGN.md picked.  Encode:
 * "enc_delta" (pass-1 variant: 1 = row-delta, 0 = general, -1 = by row width), "enc_dtile" (bytes per row-delta tile, a
 * power of two >= 2048; 0 = by input size), "enc_p2_rows" (rows per pass-2 tile of the general path, 0 = automatic;
 * the row-delta path writes every row from its own records and has no tiles), "small_sort_max" (largest dictionary
 * ranked by the tile-sort path instead of the radix sort), "sort_radix_items" (records per thread
 * in the radix passes: 4 or 16, 0 = by size), "ht_initial_log2" (first-try size of the string hash set).  Decode:
 * "dec_delta" (0/1: rows of wide schemas are assembled from the row before), "dec_strip_rows" (rows per strip of the row
 * kernels, 0 = automatic), "dec_group_lanes" (lanes per row in the narrow-schema kernels: 8, 16, 32, 0 = by schema
 * width), "dec_tile_bytes" (row-stream bytes per CTA in the row-boundary discovery).  Both: "copy_gate" (0/1, default
 * 1: host<->device copies of 8 MiB and more
 * take turns with those of the process's other contexts on the same device instead of sharing the link),
 * "kernel_timing" (0/1).  Merge: "merge_max_refs" (most referenced entries zdwb_merge_codes accepts, default and
 * ceiling 2^32 - 1; lower values let a test reach ZDWB_ERR_UNSUPPORTED).  Returns ZDWB_ERR_BAD_ARG for unknown names. */
int zdwb_ctx_set_tuning(zdwb_ctx* ctx, const char* name, long long value);

/* Number of kernels this context has launched so far (bench.py reports the delta as gpu_launches). */
unsigned long long zdwb_ctx_kernel_launches(const zdwb_ctx* ctx);

/* With the tuning knob "kernel_timing" = 1 every kernel launch is bracketed by CUDA events on the launching
 * stream.  This call synchronises, writes one line "name<TAB>launches<TAB>total_ms" per kernel into buf
 * (NUL-terminated, truncated to cap), clears the record and returns the untruncated length. */
size_t zdwb_ctx_kernel_times(zdwb_ctx* ctx, char* buf, size_t cap);

int zdwb_abi_version(void);

/* Number of CUDA devices this process can use (0 = none; the host tools spread whole ZDW blocks over them, SURVEY 8(e)). */
int zdwb_device_count(void);

/* ---- schema ---------------------------------------------------------------------------------- */

typedef struct {
  uint32_t ncols;
  const uint8_t* types; /* ncols type ids (host memory), as produced by ReadDescFile (ConvertToZDW.cpp:91-162) */
} zdwb_schema;

/* ---- encode ---------------------------------------------------------------------------------- */

typedef struct {
  int32_t trim_trailing_spaces; /* -t : ConvertToZDW.cpp:295-313 */
  int32_t input_on_device;      /* `tsv` is a device pointer (already resident in HBM) */
  int32_t output_on_device;     /* leave the encoded block in HBM: out->bytes is then a device pointer */
  int32_t more_input_follows;   /* the buffer is a window of a larger input: an unterminated last line is NOT the dropped
                                   final line of getnextrow.cpp:67-69 but the head of a row that continues in the next
                                   window; it is left unconsumed (tsv_consumed points at it) and isLast is written as 0 */
  uint32_t prev_longest_line;   /* m_LongestLine carried in from earlier blocks of the file (0 = 16384 start value,
                                   ConvertToZDW.cpp:965; the field is cumulative, getnextrow.cpp:57-65) */
  uint32_t spill_cols;          /* with max_rows: the first spill_cols columns of the row AFTER the block's last row also go
                                   through pass 1 - their strings enter this block's dictionary, their numbers its column
                                   ranges - and that row's length counts for longestLine; the row itself is not part of
                                   the block.  This is the reference's interrupted row when it runs low on memory
                                   (ConvertToZDW.cpp:334-355,404-413; stringheap.cpp:75-86; SURVEY App. B-14): with
                                   (max_rows, spill_cols) per block any file the reference cut on its own can be
                                   reproduced byte for byte.  0 = none. */
  uint64_t max_rows;            /* 0 = every row in the buffer; else close the block after this many rows */
  uint32_t heap_blocks;         /* K > 0 (and max_rows == 0): close the block where the REFERENCE would when its process is found
                                   over --mem-limit at the K-th allocation of a 64 MiB string-heap block: new strings are packed
                                   in first-occurrence order like StringHeap::copyToHeap (stringheap.cpp:31-59,75-86), the block
                                   ends in front of the row - and behind the column - whose insert opens heap block K
                                   (ConvertToZDW.cpp:334-355,404-413; SURVEY App. B-14).  K is the one number of that cut which
                                   depends on the reference's process instead of the input.  If the buffer ends before heap
                                   block K opens and more input follows, nothing is encoded (nrows = 0, tsv_consumed = 0): the
                                   caller widens the window.  K = 1 is the reference's OUT_OF_MEMORY (ZDWB_ERR_OOM). */
  uint32_t reserved_e;
} zdwb_encode_opts;

typedef struct {
  const uint8_t* bytes;   /* the block: numRows u32 | longestLine u32 | isLast u8 | dictionary | columnSize[nc] |
                             columnBase u64[#used] | rows   (SURVEY Appendix A).  isLast is 1 iff the call consumed
                             every row of the buffer; the host stitcher may patch it (offset 8). */
  size_t len;
  uint32_t nrows;         /* rows encoded into this block */
  uint32_t longest_line;  /* value written to the block header (cumulative with prev_longest_line) */
  uint64_t tsv_consumed;  /* bytes of `tsv` covered by this block (start of the next block's first row) */
  uint64_t rows_in_buffer;/* total logical rows found in the buffer */
  uint32_t bad_row;       /* ZDWB_ERR_WRONG_COLUMNS: 1-based row number ("Row %u had the problem") */
  uint32_t ncols_used;    /* columns with columnSize != 0 */
  uint64_t dict_entries;  /* unique strings in the block dictionary (Dictionary::getNumEntries) */
  uint64_t dict_bytes;    /* Dictionary::getSize(): 1 + sum(len+1) */
  uint32_t dict_index_size; /* Dictionary::getBytesInOffset() */
  uint32_t reserved;
} zdwb_block_out;

/* Encodes rows of the TSV buffer `tsv[0..n)` (which must start at a row boundary) into one ZDW block.
 * An input with zero rows yields ZDWB_OK with out->len == 0 and out->nrows == 0 ("Empty data file",
 * ConvertToZDW.cpp:824-835). */
int zdwb_encode_block(zdwb_ctx* ctx, const zdwb_schema* schema, const void* tsv, size_t n,
                      const zdwb_encode_opts* opts, zdwb_block_out* out);

/* ---- decode ---------------------------------------------------------------------------------- */

/* constant text for an output position (virtual_export_basename, UnconvertFromZDW.cpp:1253-1255) */
typedef struct {
  uint32_t pos;              /* output position */
  uint32_t len;
  const char* text;          /* host memory, no separators inside */
} zdwb_fill;

typedef struct {
  int32_t input_on_device;   /* `zdw` is a device pointer */
  int32_t output_on_device;  /* leave the TSV (and row offsets) in HBM */
  int32_t want_row_offsets;  /* also return out->row_off[nrows+1] (needed by the row-at-a-time getRow API) */
  int32_t at_end_of_file;    /* `avail` reaches the end of the file (mirrors input->eof(), UnconvertFromZDW.cpp:1577) */
  uint8_t separator;         /* '\t' (files, BufferedOutput) or '\0' (BufferedOutputInMem); the row terminator is
                                '\n' resp. '\0' */
  uint8_t reserved[7];
  /* Column projection (UnconvertFromZDW_Base::outputColumns, UnconvertFromZDW.cpp:1113-1190).  NULL = every column
   * in file order.  Otherwise out_col[c] is the output position of file column c or -1 to drop it, and n_out is the
   * number of output positions (positions no file column maps to are written as empty fields, the
   * PROVIDE_EMPTY_MISSING_COLUMNS case). */
  const int32_t* out_col;
  uint32_t n_out;
  uint32_t n_fills;          /* constant texts for positions no file column maps to */
  const zdwb_fill* fills;
  int32_t rownum_pos;        /* output position of the running row number (virtual_export_row, :1256-1261), -1 = none;
                                only honoured when out_col != NULL */
  int32_t validate_only;     /* -t: walk every row, bounds-check dictionary offsets, produce no text (:1488-1572) */
  uint64_t first_row_number; /* number of the block's first row (1-based, runs on across blocks) */
  int32_t want_flag_counts;  /* -s: also return out->flag_counts[ncols_used] = rows in which the column's bit is set */
  int32_t skim_only;         /* only find where the block ends: out->consumed (and the header fields) are filled in, no row is
                                formatted.  The file has no block length (UnconvertFromZDW.cpp:782-810,1577-1589): a host that
                                spreads blocks over several GPUs skims block k to learn where block k+1 starts (SURVEY 8(e)) */
} zdwb_decode_opts;

typedef struct {
  const uint8_t* tsv;       /* decoded rows, fields separated by `separator` */
  size_t len;
  const uint64_t* row_off;  /* nrows+1 offsets into tsv (only if want_row_offsets) */
  uint32_t nrows;           /* numRows of the block header */
  uint32_t line_length;     /* exportFileLineLength of the block header */
  uint8_t is_last;          /* isLastBlock */
  uint8_t reserved[7];
  uint64_t consumed;        /* bytes of `zdw` this block occupied: the next block starts at zdw + consumed */
  uint64_t dict_bytes;
  uint32_t ncols_used;
  uint32_t reserved2;
  const uint64_t* flag_counts; /* host memory, ncols_used entries (only if want_flag_counts) */
} zdwb_rows_out;

/* Decodes the block that starts at zdw[0] (the numRows field) given `avail` bytes. `version` is the file's
 * version word (9, 10 or 11: the block layout is identical). */
int zdwb_decode_block(zdwb_ctx* ctx, const zdwb_schema* schema, const void* zdw, size_t avail,
                      const zdwb_decode_opts* opts, zdwb_rows_out* out);

/* ---- columnar decode (ABI 5) -----------------------------------------------------------------
 * zdwb_decode_columns decodes one block, like zdwb_decode_block, into an n_cols x nrows int64 matrix on the device: row k
 * of the matrix (values + k * nrows) is file column cols[k].  A cell holds what readNextRow would print for it
 * (UnconvertFromZDW.cpp:1349-1453), as a number.  With v the column's stored value and base its columnBase:
 *   text-like (VARCHAR, TEXT, TINY/MEDIUM/LONGTEXT, DATETIME, CHAR_2, DECIMAL): the code of the string, i.e. the 0-based
 *       index of the dictionary entry at offset v + base; -1 when v == 0 (the empty string; "0.000000000000" for DECIMAL).
 *   unsigned integers: the bits of (v ? v + base : 0) (read them as uint64).
 *   signed integers: (int64)(v ? v + base : 0).  INT64_MIN is INT64_MIN (its text is the reference's quirky one).
 *   CHAR: the stored tuple (v ? v + base : 0): the low byte is the character, bits 8-15 the escaped one when the low byte
 *       is '\\'; no character when the low byte is 0.
 *   a column that is not used in the block (columnSize 0): -1 for text-like types, 0 for the others.
 * The dictionary of a block is sorted bytewise (the reference's strcmp order), so within a block codes compare like the
 * strings they stand for.  Codes belong to their block.  When a text-like column is selected the call also returns the
 * dictionary: `dict` (dict_bytes bytes, the origin NUL byte included) and `entry_off` (dict_entries + 1 offsets; entry i
 * is dict[entry_off[i] .. entry_off[i+1] - 1), entry_off[dict_entries] = dict_bytes).  Otherwise both are NULL and
 * dict_entries is 0.
 * Errors are those of zdwb_decode_block (ZDWB_ERR_TRUNCATED / ROW_COUNT / CORRUPT, with the same at_end_of_file rule),
 * plus ZDWB_ERR_CORRUPT for a selected text-like column whose offset is not the start of a dictionary entry (past the
 * dictionary, or the byte in front is not NUL: the TSV decoder prints the string's tail then, which no code expresses),
 * and ZDWB_ERR_BAD_ARG for an empty column list, an index >= ncols or an index listed twice.
 * Every output is device memory owned by the context, valid until the next call on it. */
typedef struct {
  int32_t input_on_device;   /* `zdw` is a device pointer */
  int32_t at_end_of_file;    /* `avail` reaches the end of the file (as zdwb_decode_opts.at_end_of_file) */
  const uint32_t* cols;      /* host memory: the file columns to decode, in the order of the output rows */
  uint32_t n_cols;
  uint32_t reserved;
} zdwb_columns_opts;

typedef struct {
  const int64_t* values;     /* device: n_cols x nrows */
  const uint8_t* dict;       /* device: the block's dictionary (NULL when no text-like column is selected) */
  const uint64_t* entry_off; /* device: dict_entries + 1 offsets into dict (NULL when dict is) */
  uint64_t dict_entries;
  uint64_t dict_bytes;       /* the dictionary's size, origin byte included */
  uint64_t consumed;         /* bytes of `zdw` this block occupied: the next block starts at zdw + consumed */
  uint32_t nrows;            /* numRows of the block header */
  uint32_t line_length;      /* exportFileLineLength of the block header */
  uint8_t is_last;           /* isLastBlock */
  uint8_t reserved[3];
  uint32_t ncols_used;       /* columns with columnSize != 0 */
} zdwb_columns_out;

int zdwb_decode_columns(zdwb_ctx* ctx, const zdwb_schema* schema, const void* zdw, size_t avail,
                        const zdwb_columns_opts* opts, zdwb_columns_out* out);

/* ---- merged dictionaries (ABI 5) -------------------------------------------------------------
 * zdwb_merge_codes takes n_parts parts, each a dictionary laid out as zdwb_columns_out's (dict, entry_off) plus codes
 * into it, and returns one dictionary for all of them and the codes re-coded into it:
 *   - The merged dictionary holds exactly the distinct strings that at least one code references, in strictly
 *     increasing bytewise order (memcmp over the shorter string, then the length: strcmp's order for strings without
 *     NUL).  Strings that are only in an input dictionary, with no code pointing at them, are left out.  So every code
 *     0..entries-1 occurs, codes compare like their strings, and two output codes are equal iff their strings are equal.
 *   - out->codes holds the sum of the parts' n codes, the parts in order; -1 stays -1.
 *   - The parts may come from any blocks, any columns and any files: the parts of one column over all blocks give that
 *     column a file-wide dictionary; the parts of two columns give them one shared dictionary (what a join needs).
 *   - The referenced entries of every part must be strictly increasing bytewise (a block's dictionary is).
 * Outputs are device memory owned by the context and stay valid until its next call.  With no referenced entry, dict
 * is NULL, entries and dict_bytes are 0 and entry_off holds the one offset 0; codes is NULL when n is 0.
 * Errors (each checked before any string byte is read through the offsets involved; the context works normally at its
 * next call):
 *   ZDWB_ERR_BAD_ARG: n_parts > 0 with NULL parts; a part with n > 0 and NULL codes, or with entries > 0 and a NULL dict
 *     or entry_off; a code < -1 or >= its part's entries; a referenced entry e whose offsets are not
 *     entry_off[e] < entry_off[e+1] <= dict_bytes; a part whose referenced entries are not strictly increasing bytewise.
 *   ZDWB_ERR_UNSUPPORTED: more than 2^32 - 1 referenced entries in total (counted once per part that references them).
 * The input memory must hold its final contents when the call is made: the context's stream does not wait for other
 * streams.  Device scratch: 88 bytes per referenced entry plus 4 bytes per input entry (DESIGN 4.6). */
typedef struct {
  const uint8_t*  dict;       /* device: a dictionary laid out as zdwb_columns_out.dict (NULL iff entries == 0) */
  const uint64_t* entry_off;  /* device: entries + 1 offsets; entry i = dict[entry_off[i] .. entry_off[i+1] - 1) */
  uint64_t entries;
  uint64_t dict_bytes;
  const int64_t*  codes;      /* device: n codes into this dictionary, -1 = no value */
  uint64_t n;
} zdwb_code_part;

typedef struct {
  const int64_t*  codes;      /* device: sum(n) codes, parts in order, into the merged dictionary; -1 stays -1 */
  const uint8_t*  dict;       /* device: origin NUL byte, then every entry NUL-terminated (NULL iff entries == 0) */
  const uint64_t* entry_off;  /* device: entries + 1 offsets, entry_off[entries] = dict_bytes */
  uint64_t entries;
  uint64_t dict_bytes;
  uint64_t n;
} zdwb_merge_out;

int zdwb_merge_codes(zdwb_ctx* ctx, const zdwb_code_part* parts, uint32_t n_parts, zdwb_merge_out* out);

/* ---- columns back to rows (ABI 5) ---------------------------------------------------------------
 * zdwb_render_columns writes schema->ncols columns of n rows each (cols[k] is column k, of type schema->types[k]) as TSV
 * rows: fields separated by '\t', every row ended by '\n'.  The text of every cell is the one that zdwb_encode_block (and
 * convertDWfile) reads back as the same cell, so encoding the output gives a block whose zdwb_decode_columns cells are
 * the input's (text-like cells as codes into that block's own dictionary).  cols[k] is laid out as a zdwb_merge_codes
 * part: for a text-like column codes into (dict, entry_off, entries, dict_bytes), as zdwb_columns_out / zdwb_merge_out
 * give them, -1 = no value; for any other column the int64 cells as zdwb_decode_columns gives them, and the dictionary
 * fields are ignored (NULL / 0).  Columns may share a dictionary.  The cell texts:
 *   text-like    code -1: empty (DECIMAL too: "0.000000000000" would encode as a dictionary string); code c: entry c
 *   unsigned     the decimal of the uint64 bits
 *   signed       the decimal of the int64 (INT64_MIN as "-9223372036854775808", not the decoder's lltoa text)
 *   CHAR         0: empty; sx(b) with b not NUL, '\t', '\n', '\\': the byte b; '\\' + sx(b) * 256 with b not NUL: '\\' then b
 *                (sx = signed-char extension, as the encoder computes a CHAR value)
 * out->tsv is device memory in a buffer of the context that no other entry point re-uses (as zdwb_fd_to_device's): it
 * stays valid until the next zdwb_render_columns call on the context, so it can be handed to zdwb_encode_block with
 * input_on_device = 1.  Zero rows: ZDWB_OK with len 0.
 * ZDWB_ERR_BAD_ARG (zdwb_last_error names the lowest (column, row) at fault and the rule): NULL arguments, zero columns,
 *   columns of different n, a type the encoder does not know (4, 5: the VISID types); a code < -1 or >= entries; a
 *   referenced entry whose offsets are not entry_off[e] < entry_off[e+1] <= dict_bytes, that is empty, holds a NUL or does
 *   not end in one, holds a '\t' or '\n' not preceded by an odd run of backslashes, or ends in an odd run of backslashes
 *   (the row reader would not give it back as one field); a CHAR value of none of the forms above; an empty cell in a
 *   table of one column (the row "\n" would be skipped).  Entries no code references are not checked for content, and
 *   nothing is read through an entry's offsets before they are checked.  ZDWB_ERR_UNSUPPORTED: 2^36 rows or 2^24
 *   columns and more.  The context works normally at its next call.
 * The input memory must hold its final contents when the call is made: the context's stream does not wait for other
 * streams.  Device scratch: 8 bytes per row and 1 byte per entry of every distinct dictionary (DESIGN 4.7). */
typedef struct {
  const uint8_t* tsv;   /* device: the rows; fields separated by '\t', every row ended by '\n' */
  uint64_t len;
} zdwb_render_out;

int zdwb_render_columns(zdwb_ctx* ctx, const zdwb_schema* schema, const zdwb_code_part* cols, zdwb_render_out* out);

/* ---- predicates over a dictionary (ABI 5) -------------------------------------------------------
 * Both calls take a dictionary as a zdwb_code_part whose codes and n are ignored: a merged one (zdwb_merge_out) or a
 * block's (zdwb_columns_out).  Entry i is dict[entry_off[i] .. entry_off[i+1] - 1).  A filter on a text column is then
 * one pass over its distinct strings plus one gather of the per-entry answer by the codes.
 *
 * zdwb_match_like: SQL LIKE of every entry against opts->pattern, and of opts->null_text, the text that code -1 stands
 *   for ("" for text columns, "0.000000000000" for DECIMAL).  out->flags holds entries + 1 bytes, 1 = match: one per
 *   entry, the last one for null_text.  The whole entry is matched, bytewise, as it is stored (what unconvertDWfile prints
 *   for the cell, TSV escapes included): '%' matches any run of bytes, the empty one too; '_' matches exactly one BYTE
 *   (not one UTF-8 character); the escape byte followed by any byte matches that byte; every other byte matches itself.
 *   With ignore_case the ASCII letters A-Z / a-z match either case (escaped ones too); no other byte is folded.
 * zdwb_find_strings: for the n query strings in queries (query i = bytes[off[i] .. off[i+1]), device memory),
 *   out->rank[i] is the number of entries bytewise less than query i (lower_bound, in [0, entries]) and out->found[i] is
 *   1 iff entry rank[i] equals it.  The entries must be strictly increasing bytewise (memcmp over the shorter string, then
 *   the length: the order of zdwb_merge_codes and of a block's dictionary); every entry is checked against the one
 *   before it.  Queries may be unsorted, repeated, empty, and hold any byte.  rank and found are NULL when n is 0.
 * Outputs are device memory owned by the context and stay valid until its next call.  The input memory must hold its
 * final contents when the call is made: the context's stream does not wait for other streams.
 * Errors (checked before anything is read through the offsets involved; zdwb_last_error names the lowest entry or query
 * at fault; the context works normally at its next call):
 *   ZDWB_ERR_BAD_ARG: a NULL dict, opts, queries or out; entries > 0 with a NULL dict or entry_off; a pattern or null_text
 *     with a length and a NULL pointer; escape not in -1 .. 255; a pattern that ends in a lone escape byte; an entry whose
 *     offsets are not entry_off[e] < entry_off[e+1] <= dict_bytes; (find) n > 0 with NULL off, bytes_len > 0 with NULL
 *     bytes, an entry not greater than the one before it, a query whose offsets are not off[i] <= off[i+1] <= bytes_len.
 *   ZDWB_ERR_UNSUPPORTED: a pattern of 2^32 - 1 bytes or more.
 * Device scratch: match 2 bytes per pattern byte; find 16 bytes per entry (DESIGN 4.8). */
typedef struct {
  const uint8_t* pattern;    /* host memory */
  uint64_t pattern_len;
  const uint8_t* null_text;  /* host memory: the text of code -1 */
  uint64_t null_text_len;
  int32_t escape;            /* -1 = no escape byte, else 0 .. 255 */
  int32_t ignore_case;       /* fold ASCII A-Z / a-z */
} zdwb_like_opts;

typedef struct {
  const uint8_t* flags;      /* device: n bytes, 0 / 1; flags[entries] is null_text's */
  uint64_t n;                /* entries + 1 */
} zdwb_match_out;

typedef struct {
  const uint8_t* bytes;      /* device: the query strings back to back */
  uint64_t bytes_len;
  const uint64_t* off;       /* device: n + 1 offsets into bytes */
  uint64_t n;
} zdwb_strings;

typedef struct {
  const int64_t* rank;       /* device: n lower bounds */
  const uint8_t* found;      /* device: n bytes, 1 iff entry rank[i] equals query i */
  uint64_t n;
} zdwb_find_out;

int zdwb_match_like(zdwb_ctx* ctx, const zdwb_code_part* dict, const zdwb_like_opts* opts, zdwb_match_out* out);
int zdwb_find_strings(zdwb_ctx* ctx, const zdwb_code_part* dict, const zdwb_strings* queries, zdwb_find_out* out);

/* ---- numbers from and to text (ABI 5) -----------------------------------------------------------
 * ZDW stores DATETIME and DECIMAL cells as dictionary strings.  These two calls turn a dictionary into numbers, once per
 * distinct string, and numbers back into a dictionary, so that torch can compute on time and money columns.
 *
 * zdwb_parse_numbers: the number of every entry of `dict` (taken as by zdwb_match_like: codes and n are ignored) and of
 *   opts->null_text, the text of code -1 ("" for text columns, "0.000000000000" for DECIMAL, as zdwb_like_opts).  Every
 *   text is parsed as it is stored, bytewise: no white space is allowed and nothing is trimmed.  out->values[e] is the
 *   number and out->ok[e] is 1 when the text is in the grammar and its number fits, else both are 0.  The last element is
 *   null_text's.
 *   DATETIME: "YYYY-MM-DD HH:MM:SS", optionally followed by '.' and 1 to 6 digits, or "YYYY-MM-DD" alone (midnight).
 *     Every field has exactly the digits shown.  Dates run from 0001-01-01 to 9999-12-31 on the proleptic Gregorian
 *     calendar; hours are 0-23, minutes and seconds 0-59; no time zone is applied.  So "0000-00-00 00:00:00",
 *     "24:00:00" and "1900-02-29" are not ok.  The value is microseconds since 1970-01-01 00:00:00 (negative before).
 *   DECIMAL of scale s = opts->digits: [+-]?(D+(\.D*)?|\.D+) with D an ASCII digit; no exponent.  The value is the number
 *     times 10^s and must be exact (fraction digits past the s-th are '0') and lie in [INT64_MIN, INT64_MAX].  Leading
 *     zeros and trailing fraction zeros never overflow.  Scale 0 reads the integers a VARCHAR column holds.
 * zdwb_format_numbers: the inverse, for n values that are strictly increasing (as torch.unique returns them; every value
 *   is checked against the one before it).  out is a dictionary laid out as zdwb_merge_out's: dense, entries strictly
 *   increasing bytewise, out->codes[i] the code of values[i]'s text, out->n = n.  So (codes, dict, entry_off) is a row of a
 *   ColumnTable and its dictionary, fit for zdwb_render_columns, zdwb_match_like, zdwb_find_strings and zdwb_merge_codes.
 *   DATETIME: "YYYY-MM-DD HH:MM:SS", then '.' and exactly opts->digits fraction digits when digits > 0.
 *   DECIMAL: an optional '-', the integer digits without leading zeros ("0" when the integer part is zero), then '.' and
 *     exactly opts->digits digits when digits > 0.  INT64_MIN is written as every other value is.
 *   Parsing a formatted text with the same opts gives the value back.  With n == 0: dict and codes are NULL, entries and
 *   dict_bytes 0, and entry_off holds the one offset 0.
 * Outputs are device memory owned by the context and stay valid until its next call.  The input memory must hold its
 * final contents when the call is made: the context's stream does not wait for other streams.
 * Errors (checked before anything is read through the offsets involved; zdwb_last_error names the lowest entry or value at
 * fault; the context works normally at its next call):
 *   ZDWB_ERR_BAD_ARG: NULL arguments; a kind that is neither ZDWB_NUM_DATETIME nor ZDWB_NUM_DECIMAL; digits outside 0..18
 *     (DECIMAL) or, in format, 0..6 (DATETIME); null_text_len > 0 with a NULL null_text; entries > 0 with a NULL dict or
 *     entry_off; (parse) an entry whose offsets are not entry_off[e] < entry_off[e+1] <= dict_bytes; (format) n > 0 with
 *     NULL values, a value not greater than the one before it, a DATETIME outside 0001-01-01 00:00:00 ..
 *     9999-12-31 23:59:59.999999 or not a multiple of 10^(6 - digits) microseconds.
 *   ZDWB_ERR_UNSUPPORTED: (format) texts of 2^32 bytes or more in all, each counted with its NUL terminator (the limit of
 *     the string sort).
 * Device scratch: parse null_text_len + 24 bytes; format 20 bytes per value, the texts with their terminators, and the
 * string sort's own: 40 bytes per value, plus up to 20 per value still tied after the first 8 bytes (DESIGN 4.9). */
enum { ZDWB_NUM_DATETIME = 0, ZDWB_NUM_DECIMAL = 1 };

typedef struct {
  int32_t kind;              /* ZDWB_NUM_DATETIME or ZDWB_NUM_DECIMAL */
  int32_t digits;            /* DECIMAL: the scale, 0..18.  DATETIME: ignored by parse; format: fraction digits, 0..6 */
  const uint8_t* null_text;  /* parse only, host memory: the text of code -1 */
  uint64_t null_text_len;
} zdwb_number_opts;

typedef struct {
  const int64_t* values;     /* device: n numbers; values[entries] is null_text's */
  const uint8_t* ok;         /* device: n bytes, 1 = the text is in the grammar and its number fits */
  uint64_t n;                /* entries + 1 */
} zdwb_parse_out;

int zdwb_parse_numbers(zdwb_ctx* ctx, const zdwb_code_part* dict, const zdwb_number_opts* opts, zdwb_parse_out* out);
int zdwb_format_numbers(zdwb_ctx* ctx, const int64_t* values, uint64_t n, const zdwb_number_opts* opts,
                        zdwb_merge_out* out);

/* ---- pinned host staging (used by the host classes and the end-to-end bench) ------------------ */
void* zdwb_host_alloc(size_t bytes);   /* cudaHostAlloc'd (pinned, usable from every device) memory, NULL on failure */
void zdwb_host_free(void* p);

/* ---- file descriptor <-> device (ABI 4) ---------------------------------------------------------
 * What the host tools use instead of window-sized host buffers: the reference reads its input with fgets
 * (getnextrow.cpp:26-84) and writes rows through BufferedOutput (BufferedOutput.cpp:239-260); here a window of the
 * input file goes straight to the device and the decoded rows of a block straight to the output file, in 8 MiB chunks
 * through a pinned ring owned by the context, the copy of one chunk under the read / write of the next.
 *   zdwb_fd_to_device: `len` bytes of fd from `offset` (pread; offset < 0: read() at the descriptor's position) into a
 *     device buffer of the context; *dev stays valid until the next zdwb_fd_to_device call on it.  Encode it with
 *     zdwb_encode_opts.input_on_device = 1.
 *   zdwb_device_to_fd: `len` device bytes (e.g. zdwb_rows_out.tsv of a call with output_on_device = 1) to fd at `offset`
 *     (pwrite; offset < 0: write()).  Returns when everything is written.
 * ZDWB_ERR_BAD_ARG with zdwb_last_error() set when the descriptor fails or ends early. */
int zdwb_fd_to_device(zdwb_ctx* ctx, int fd, long long offset, size_t len, const void** dev);
int zdwb_device_to_fd(zdwb_ctx* ctx, const void* dev, size_t len, int fd, long long offset);

#ifdef __cplusplus
}
#endif
#endif /* ZDW_B200_H */
