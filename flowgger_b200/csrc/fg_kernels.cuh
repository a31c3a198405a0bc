// fg_kernels.cuh — launch parameters shared by fg_kernels.cu and fg_abi.cu
#pragma once
#include <stdint.h>
#ifdef FG_HOST_EMU
#include "../../tests/emu/cuda_shim.h"
#else
#include <cuda_runtime.h>
#endif

namespace fg {

// LTSV decoder configuration in device memory (ltsv_decoder.rs:19-22)
struct LtsvDeviceConfig {
    int32_t has_schema;
    int32_t n_schema;
    const uint8_t* names;       // concatenated schema key bytes
    const int32_t* name_off;    // [n_schema+1]
    const int32_t* types;       // [n_schema] fg_ltsv_type
    const uint8_t* suffix;      // concatenated suffix bytes
    int32_t suffix_off[6];      // per fg_ltsv_type: [t]..[t+1]; empty span + present bit
    uint32_t suffix_present;    // bit t set if a suffix is configured for type t
};

// RFC3164: zone database behind time_tz::timezones::get_by_name (rfc3164_decoder.rs:196), packed by fg_tz.cu.
// A zone is a run of spans; span j is in force from LOCAL second key[j] on (key of a zone's first span: INT64_MIN), see
// fg_rfc3164.cuh: tz_offset_local.
struct TzDeviceTable {
    int32_t n_names;            // identifiers (0: no database: no token is a zone name)
    int32_t min_len, max_len;   // of the identifiers
    uint32_t first_mask[8];     // bit c: some identifier starts with byte c
    const unsigned long long* hash;  // [n_names] FNV-1a 64 of the identifier, ascending
    const int32_t* zone;        // [n_names] zone of the identifier (links share the zone of their target)
    const int32_t* name_off;    // [n_names + 1] into names, in hash order
    const uint8_t* names;
    const int32_t* first;       // [zones + 1] span range of a zone
    const long long* key;       // [spans]
    const int32_t* off;         // [spans] UTC offset in seconds
};
struct R3164DeviceConfig {
    int32_t year;               // OffsetDateTime::now_utc().year() (rfc3164_decoder.rs:175), fixed per call
    TzDeviceTable tz;
    uint8_t* arena;             // re-joined messages (rfc3164_decoder.rs:67: tokens joined by one space)
    uint32_t arena_cap;
    uint32_t* arena_counter;    // bump allocator; keeps counting past arena_cap (the host regrows and redoes the batch)
};

struct ParseParams {
    const uint8_t* bytes;     // device copy of the caller's byte buffer (base of all spans)
    const int32_t* offsets;   // [n+1] line offsets into bytes
    int32_t n;                // lines in this launch
    int32_t line0;            // batch index of the first line of this launch
    int32_t tile_bytes;       // dynamic shared memory staging tile, multiple of 16
    // row columns, element 0 = first line of this launch
    double* ts;
    uint32_t* meta;
    int2* host;
    int2* app;
    int2* proc;
    int2* msgid;
    int2* msg;
    int2* full;
    int2* sd;
    // structured-data side table
    int2* entry_name;
    unsigned long long* entry_val;
    uint8_t* entry_meta;
    // provisional rows of a line, indexed by its byte offset (see Format<>::scratch_index)
    int2* tmp_name;
    unsigned long long* tmp_val;
    uint8_t* tmp_meta;
    // split mode (fg_split_decode): every line still carries its "\n" / "\r\n" terminator, and lines flagged invalid
    // by the UTF-8 pass are not parsed
    const uint8_t* line_invalid;  // [n] or nullptr
    int32_t strip_eol;
    uint32_t* entry_counter;  // running total (atomic bump, one add per CTA round)
    uint32_t entry_cap;
    const uint32_t* bad_offsets;  // set by check_offsets_kernel when the offsets array is not monotone / in range: kernels do nothing
    // GELF: launch-relative numbers of the lines the fast walker hands to the exact parser (post_gelf_kernel)
    uint32_t* slow_list;
    uint32_t* slow_count;
    LtsvDeviceConfig ltsv;
    R3164DeviceConfig r3164;
};

// ---- RFC5424 fast path (fg_parse5424.cu) ------------------------------------------------------------------------
// compact row, 32 bytes per line (include/flowgger_cuda.h: fg_row5424)
struct Row5424 {
    double ts;
    uint32_t meta;      // status | facility << 8 | severity << 16 | flags << 24
    uint32_t sd_first;  // first 8-byte entry of this line (FG_FLAG_WIDE: index into the wide rows instead)
    uint16_t sd_count;  // entries of this line (headers + pairs + extension rows)
    uint16_t sp[5];     // spaces 2..6 relative to the line start
    uint16_t msg_off, msg_len;
};
static_assert(sizeof(Row5424) == 32, "Row5424 must be 32 bytes");
// wide row (fg_wide_row): absolute spans like the LTSV / GELF columns
struct WideRow {
    int32_t line;
    uint32_t meta;
    double ts;
    int2 host, app, proc, msgid, msg, full, sd;  // sd = {first wide entry, count}
};
static_assert(sizeof(WideRow) == 72, "WideRow must be 72 bytes");

enum { K5_ENTRIES = 0, K5_ARENA = 1, K5_WIDE_ROWS = 2, K5_WIDE_ENTRIES = 3, K5_ESC_LIST = 4, K5_WIDE_LIST = 5, K5_BAD_OFFSETS = 6, K5_COUNT = 8 };

struct Parse5424Params {
    const uint8_t* bytes;
    const int32_t* offsets;  // [n+1], element 0 = first line of this launch
    int32_t n;
    int32_t tile_bytes;      // staging tile (multiple of 512); the bitmap (tile_bytes / 8 + 16 bytes) follows it
    uint4* rows;             // 2 x uint4 per line, element 0 = first line of this launch
    unsigned long long* entries;
    uint32_t entry_cap;
    uint32_t* counters;      // K5_*: ENTRIES / ARENA / WIDE_* run over the whole batch, the two LIST lengths are per launch
    uint32_t* esc_list;      // launch-relative line numbers with escaped values
    uint32_t* wide_list;     // launch-relative line numbers for the wide kernel
    uint8_t* arena;
    uint32_t arena_cap;
    WideRow* wide_rows;
    uint32_t wide_cap;
    int2* wentry_name;
    unsigned long long* wentry_val;
    uint8_t* wentry_meta;
    uint32_t wentry_cap;
    int32_t line0;           // batch index of the first line of this launch (WideRow.line)
    const uint32_t* bad_offsets;  // see ParseParams
    const uint8_t* line_invalid;  // split mode, or nullptr
    int32_t strip_eol;
};

// parse5424_kernel + post5424_kernel; when given, the two events bracket the parse kernel alone (roofline measurement)
cudaError_t launch_parse5424(const Parse5424Params& p, cudaStream_t stream, cudaEvent_t dom0 = nullptr, cudaEvent_t dom1 = nullptr);
cudaError_t configure_parse5424(int max_tile_bytes);
int parse5424_smem_bytes(int tile_bytes);

// ---- fused GELF encoder over the RFC5424 results (fg_gelf_encode.cu) ---------------------------------------------------
struct GelfEncodeParams {
    const uint8_t* bytes;
    const int32_t* offsets;  // [n+1], element 0 = first line of this launch
    int32_t n;
    const uint4* rows;       // compact rows of these lines
    const unsigned long long* entries;
    const uint8_t* arena;
    const WideRow* wide_rows;
    const int2* wentry_name;
    const unsigned long long* wentry_val;
    const uint8_t* wentry_meta;
    // fixed GELF keys + output.gelf_extra, sorted by key on the host (extras already replace fixed keys of the same name)
    const uint8_t* static_blob;
    int32_t n_static;
    const int32_t* static_key_off;  // [n_static+1] raw key bytes (for ordering against the SD names)
    const int32_t* static_lit_off;  // [n_static+1] text to emit: `"key":`, for an extra `"key":"value"`
    const int32_t* static_kind;     // [n_static] GF_*
    uint32_t* lens;                 // [n] record lengths (size pass)
    uint32_t* rel;                  // [n] exclusive sum of lens inside this launch
    unsigned long long* base;       // base[0] = output bytes before this launch, base[1] receives base[0] + this launch's bytes
    uint8_t* out;
    unsigned long long out_cap;
    long long* out_offsets;         // [n+1] absolute record offsets, element 0 = first line of this launch
    uint8_t* status;                // [n] decoder status per line (0 = a record was written)
    const uint32_t* bad_offsets;
    uint32_t entry_cap, wide_cap, wentry_cap;  // a table that overflowed is not read (the batch is redone after a regrow)
    int32_t tile_bytes;                        // staging tile of the two kernels (dynamic shared memory)
};
cudaError_t configure_gelf_encode(int max_tile_bytes);
cudaError_t launch_gelf_encode(const GelfEncodeParams& p, void* d_scan_temp, size_t scan_temp_bytes, cudaStream_t stream);
size_t gelf_scan_temp_bytes(int n);

// RFC5424 (short lines, staged tile): 64-line CTAs — tile waits and barriers half as wide as with 128 lines
#ifndef FG_R5_LINES  // profiles/variants.sh builds other shapes with -DFG_R5_LINES / -DFG_R5_MINB for A/B runs
#define FG_R5_LINES 64
#endif
#ifndef FG_R5_MINB  // 16 CTAs/SM (64 registers, tile slack 2 %) measured 2 % faster than 14 (71 registers, 10 %): profiles/r2_notes.md
#define FG_R5_MINB 16
#endif
constexpr int kRfc5424LinesPerCta = FG_R5_LINES;
constexpr int kRfc5424CtasPerSm = FG_R5_MINB;
// LTSV (fg_parse_ltsv.cu): 64 lines and 256 threads per CTA; a CTA round has kLtsvStageSlots slots, one per tab-separated part
#ifndef FG_LTSV_LINES
#define FG_LTSV_LINES 64
#endif
#ifndef FG_LTSV_THREADS
#define FG_LTSV_THREADS 256
#endif
constexpr int kLtsvLinesPerCta = FG_LTSV_LINES;
constexpr int kLtsvThreadsPerCta = FG_LTSV_THREADS;
constexpr int kLtsvStageSlots = kLtsvLinesPerCta * 24;
constexpr int kLtsvMaxTile = 65024;  // tile positions are packed into 16 bits
// GELF (fg_parse_gelf.cu): 64 lines and 256 threads per CTA; a CTA round has kGelfStageSlots slots, one per top-level member
#ifndef FG_GELF_LINES
#define FG_GELF_LINES 64
#endif
#ifndef FG_GELF_THREADS
#define FG_GELF_THREADS 256
#endif
constexpr int kGelfLinesPerCta = FG_GELF_LINES;
constexpr int kGelfThreadsPerCta = FG_GELF_THREADS;
constexpr int kGelfCtasPerSm = 3;  // tile (~34 KB at 520 B/line) + bitmap + slots: 3 CTAs = 24 warps per SM
constexpr int kGelfStageSlots = kGelfLinesPerCta * 16;
constexpr int kGelfMaxTile = 65024;
// RFC3164 (fg_parse3164.cu): 64 lines and 64 threads per CTA, one thread per line over the staged tile
#ifndef FG_R3_LINES  // profiles/r2_rfc3164_variants.sh builds other shapes for A/B runs
#define FG_R3_LINES 64
#endif
#ifndef FG_R3_MINB
#define FG_R3_MINB 16
#endif
#ifndef FG_R3_LOCKSTEP  // 1: r3164_parse_lockstep (warp-wide phases), 0: r3164_parse_line (one thread on its own); fg_rfc3164.cuh
#define FG_R3_LOCKSTEP 1
#endif
constexpr int kR3164LinesPerCta = FG_R3_LINES;
constexpr int kR3164CtasPerSm = FG_R3_MINB;
constexpr int kR3164MaxTile = 65024;
constexpr int lines_per_cta(int fmt) {
    return fmt == 0 ? kRfc5424LinesPerCta : (fmt == 1 ? kLtsvLinesPerCta : (fmt == 2 ? kGelfLinesPerCta : kR3164LinesPerCta));
}

cudaError_t launch_parse(int fmt, const ParseParams& p, cudaStream_t stream);
// LTSV on the bitmap pipeline (fg_parse_ltsv.cu); launch_parse routes fmt 1 here
cudaError_t launch_parse_ltsv(const ParseParams& p, cudaStream_t stream);
cudaError_t configure_parse_ltsv(int max_tile_bytes);
int parse_ltsv_smem_bytes(int tile_bytes, bool typed);
// GELF on the bitmap pipeline + the exact parser over the slow list (fg_parse_gelf.cu); launch_parse routes fmt 2 here
cudaError_t launch_parse_gelf(const ParseParams& p, cudaStream_t stream);
cudaError_t configure_parse_gelf(int max_tile_bytes);
int parse_gelf_smem_bytes(int tile_bytes);
// RFC3164 (fg_parse3164.cu); launch_parse routes fmt 3 here
cudaError_t launch_parse3164(const ParseParams& p, cudaStream_t stream);
cudaError_t configure_parse3164(int max_tile_bytes);
// offsets[0 .. n] must be non-decreasing and within [0, max_bytes]; otherwise *flag |= 1 (the parse kernels then return at once)
cudaError_t launch_check_offsets(const int32_t* d_offsets, int n, long long max_bytes, uint32_t* d_flag, cudaStream_t stream);
cudaError_t configure_kernels(int max_tile_bytes, int max_tile5424);
const char* kernel_build_info();

// device-side line framing + UTF-8 validation (fg_split.cu)
cudaError_t launch_split_chunk(const uint8_t* d_bytes, long long nbytes, long long c0, long long c1, int is_last, uint32_t* d_seg,
                               uint32_t* d_run, int32_t* d_cum_k, int32_t* d_offsets, int32_t* d_n_lines, int max_lines,
                               uint8_t* d_invalid, int delim, cudaStream_t stream);
int split_segments(long long nbytes);

}  // namespace fg
