// fg_abi.cu — the C ABI declared in include/flowgger_cuda.h.
//
// Host side of the drop-in boundary: owns the device buffers, pinned host
// result arrays and streams of one context, pipelines host<->device copies
// with the parse kernels chunk by chunk, and exposes the device-resident
// variant used for roofline measurement.  There is no CPU parsing anywhere in
// this file: if CUDA is unavailable every entry point returns an error.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/flowgger_cuda.h"
#include "fg_kernels.cuh"
#include "fg_status.h"
#include "fg_rfc3164.cuh"
#include "fg_tz.h"

namespace {

// The reference's `&'static str` for every status (file:line in /root/reference/src/flowgger/decoder/)
const char* kErrorStrings[FG_ST_COUNT] = {};
struct ErrorTableInit {
    ErrorTableInit() {
        auto& t = kErrorStrings;
        t[FG_E5_BOM] = "Unsupported BOM";                                        // rfc5424_decoder.rs:69
        t[FG_E5_PRI_BRACKETS] = "The priority should be inside brackets";         // :76
        t[FG_E5_INVALID_PRI] = "Invalid priority";                                // :83
        t[FG_E5_MISSING_VERSION] = "Missing version";                             // :84
        t[FG_E5_UNSUPPORTED_VERSION] = "Unsupported version";                     // :86
        t[FG_E5_MISSING_TS] = "Missing timestamp";                                // :25
        t[FG_E5_BAD_TS] = "Unable to parse the date from RFC3339 to Unix time in RFC5424 decoder";  // :97
        t[FG_E5_MISSING_HOST] = "Missing hostname";                               // :26
        t[FG_E5_MISSING_APP] = "Missing application name";                        // :27
        t[FG_E5_MISSING_PROCID] = "Missing process id";                           // :28
        t[FG_E5_MISSING_MSGID] = "Missing message id";                            // :29
        t[FG_E5_MISSING_DATA] = "Missing message data";                           // :30
        t[FG_E5_MISSING_MSG] = "Missing log message";                             // :129,:148
        t[FG_E5_MALFORMED] = "Malformated RFC5424 message";                       // :154,:159
        t[FG_E5_MISSING_SD] = "Missing structured data";                          // :177
        t[FG_E5_SD_FORMAT] = "Format error in the structured data";               // :235
        t[FG_E5_SD_NO_END] = "Missing ] after structured data";                   // :239
        t[FG_E5_MISSING_PRI_VERSION] = "Missing priority and version";            // :24 (unreachable)
        t[FG_E5_EMPTY_PRI] = "Empty priority";                                    // :81 (unreachable)
        t[FG_E5_MISSING_SD_ID] = "Missing structured data id";                    // :176 (unreachable)
        t[FG_EL_TS] = "Unable to parse the English to Unix timestamp in LTSV decoder";  // ltsv_decoder.rs:252
        t[FG_EL_SEV] = "Invalid severity level";                                  // :116
        t[FG_EL_SEV_HIGH] = "Severity level should be <= 7";                      // :118
        t[FG_EL_BOOL] = "Type error; boolean was expected";                       // :143
        t[FG_EL_F64] = "Type error; f64 was expected";                            // :159
        t[FG_EL_I64] = "Type error; i64 was expected";                            // :175
        t[FG_EL_U64] = "Type error; u64 was expected";                            // :191
        t[FG_EL_MISSING_TS] = "Missing timestamp";                                // :205
        t[FG_EL_MISSING_HOST] = "Missing hostname";                               // :206
        t[FG_EG_JSON] = "Invalid GELF input, unable to parse as a JSON object";   // gelf_decoder.rs:49
        t[FG_EG_EMPTY] = "Empty GELF input";                                      // :50
        t[FG_EG_TS] = "Invalid GELF timestamp";                                   // :53
        t[FG_EG_HOST] = "GELF host name must be a string";                        // :58
        t[FG_EG_SHORT] = "GELF short message must be a string";                   // :66
        t[FG_EG_FULL] = "GELF full message must be a string";                     // :74
        t[FG_EG_VERSION_T] = "GELF version must be a string";                     // :78
        t[FG_EG_VERSION] = "Unsupported GELF version";                            // :80
        t[FG_EG_SEV] = "Invalid severity level";                                  // :83
        t[FG_EG_SEV_HIGH] = "Invalid severity level (too high)";                  // :85
        t[FG_EG_SD_TYPE] = "Invalid value type in structured data";               // :97
        t[FG_EG_MISSING_HOST] = "Missing hostname";                               // :110
        t[FG_ES_INVALID_UTF8] = "Invalid UTF-8 input";                            // splitter/line_splitter.rs:23
        t[FG_E3_PRI_MALFORMED] = "Malformed RFC3164 event: Invalid priority";     // rfc3164_decoder.rs:131
        t[FG_E3_PRI_INVALID] = "Invalid priority";                                // :137
        t[FG_E3_CUSTOM] = "Malformed RFC3164 event: Invalid timestamp or hostname";  // :120
        t[FG_E3_TIME_FORMAT] = "Invalid time format";                             // :158
        t[FG_E3_WITH_YEAR] = "Unable to parse RFC3164 date with year";            // :178
        t[FG_E3_DATE] = "Unable to parse the date in RFC3164 decoder";            // :211
        t[FG_E3_PANIC] = "(the reference panics here: index out of bounds, rfc3164_decoder.rs:64)";
    }
} g_error_table_init;

constexpr size_t kPad = 256;            // slack after the device byte buffer (16-byte bulk-copy granules)
constexpr size_t kBounceBytes = 32u << 20;  // pinned bounce buffers for pageable caller memory
constexpr size_t kL2FlushBytes = 256u << 20;
constexpr int kRedo = 1;  // drain(): tables were regrown and the attempt must be enqueued again (FG_E_* codes are negative)
const char* const kBadOffsets = "offsets must be non-decreasing and within max_batch_bytes";

// A device array, its pinned host mirror and their capacity in elements of `width` bytes.  alloc() rounds the
// capacity up to a multiple of `round` and allocates `pad` bytes more on both sides.
struct Mirror {
    const size_t width, round, pad;
    uint8_t* d = nullptr;
    uint8_t* h = nullptr;
    size_t cap = 0;

    explicit Mirror(size_t width_, size_t round_ = 1, size_t pad_ = 0) : width(width_), round(round_), pad(pad_) {}
    Mirror(const Mirror&) = delete;
    Mirror& operator=(const Mirror&) = delete;
    ~Mirror() { release(); }

    void release() {
        if (d) cudaFree(d);
        if (h) cudaFreeHost(h);
        d = h = nullptr;
        cap = 0;
    }
    cudaError_t alloc(size_t n) {
        release();
        n = (n + round - 1) / round * round;
        cudaError_t e = cudaMalloc(&d, n * width + pad);
        if (e == cudaSuccess) e = cudaHostAlloc(&h, n * width + pad, cudaHostAllocDefault);
        if (e == cudaSuccess) cap = n;
        return e;
    }
    // elements [from, to) back to the host mirror
    cudaError_t d2h(size_t from, size_t to, cudaStream_t s) const {
        if (to <= from) return cudaSuccess;
        return cudaMemcpyAsync(h + from * width, d + from * width, (to - from) * width, cudaMemcpyDeviceToHost, s);
    }
    template <class T>
    T* dev() const { return (T*)d; }
    template <class T>
    T* host() const { return (T*)h; }
};

// One result table of a format: the counter (fg::K5_*) that bounds it, the mirrors that hold it (one per column, all
// with the same capacity) and the capacity a format allocates when it finds the table empty.
struct Table {
    int slot;
    std::vector<Mirror*> cols;
    size_t first;
    bool grow_to_first;  // also grown to `first` when another format left it smaller
};

}  // namespace

static_assert(sizeof(fg_wide_row) == sizeof(fg::WideRow), "wide rows are copied back byte for byte");

struct fg_ctx {
    int device = 0;
    size_t max_bytes = 0;
    int max_lines = 0;
    int chunk_lines = 0;
    cudaStream_t s_h2d = nullptr, s_comp = nullptr, s_d2h = nullptr;
    // device: input; the host side receives the line offsets fg_split_decode finds
    uint8_t* d_bytes = nullptr;
    Mirror offsets{sizeof(int32_t)};
    uint32_t* d_k = nullptr;  // counter block (fg::K5_*)
    uint8_t* d_flush = nullptr;
    // LTSV / GELF / RFC3164: columnar rows (9 columns sized for max_lines)
    Mirror rows{1};
    // 17-byte side-table rows (LTSV / GELF, RFC5424 wide lines) + LTSV / GELF scratch
    Mirror entry_name{sizeof(fg_span), 256}, entry_val{sizeof(uint64_t), 256}, entry_meta{1, 256};
    int2* d_tmp_name = nullptr;  // provisional side-table rows, indexed by byte offset / scratch_div
    unsigned long long* d_tmp_val = nullptr;
    uint8_t* d_tmp_meta = nullptr;
    size_t tmp_cap = 0;
    // RFC5424: compact rows, 8-byte entries, work lists, arena, wide rows
    Mirror rows5{sizeof(fg_row5424)};
    Mirror e8{8, 256};
    uint32_t* d_esc_list = nullptr;
    uint32_t* d_wide_list = nullptr;  // RFC5424 wide lines, GELF slow lines
    Mirror arena{1, 256};
    Mirror wide{sizeof(fg_wide_row)};
    std::vector<Table> tables[4];  // by fg_format (list_tables)
    // fused GELF encoder (fg_decode_encode_gelf)
    uint32_t* d_enc_lens = nullptr;
    uint32_t* d_enc_rel = nullptr;
    Mirror enc_base{sizeof(unsigned long long)};  // [chunks + 1] running output size
    Mirror enc_out{1, 4096, 16};
    Mirror enc_offsets{sizeof(int64_t)};
    Mirror enc_status{1};
    void* d_scan_temp = nullptr;
    size_t scan_temp_bytes = 0;
    uint8_t* d_static_blob = nullptr;  // fixed GELF keys + output.gelf_extra, sorted
    int n_static = 0;
    const int32_t* d_static_key_off = nullptr;
    const int32_t* d_static_lit_off = nullptr;
    const int32_t* d_static_kind = nullptr;
    std::vector<std::pair<std::string, std::string>> gelf_extra;
    // split mode (fg_split_decode)
    uint32_t* d_seg = nullptr;
    int32_t* d_n_lines = nullptr;
    uint8_t* d_invalid = nullptr;
    int32_t* h_n_lines = nullptr;
    float last_split_ms = 0.f;
    cudaEvent_t ev_s0 = nullptr, ev_s1 = nullptr;
    cudaStream_t s_parse = nullptr;
    std::vector<cudaEvent_t> ev_split;
    Mirror cum{sizeof(int32_t)};
    // RFC3164: the year `now_utc().year()` stands for (0: read the clock at every call) and the zone database
    int r3164_year = 0;
    int call_year = 1970;  // the year of the call in progress (current_year())
    std::string tzdir;
    fg::TzHostTable tz_host;
    uint8_t* d_tz_blob = nullptr;
    fg::TzDeviceTable tz_dev{};
    // LTSV config blobs
    uint8_t* d_ltsv_blob = nullptr;
    fg::LtsvDeviceConfig ltsv{};
    // pinned host
    uint32_t* h_counts = nullptr;  // per-step snapshots of the counter block (fg::K5_COUNT words each)
    int h_counts_cap = 0;
    uint8_t* h_bounce[2] = {nullptr, nullptr};
    cudaEvent_t bounce_ev[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> ev_h2d, ev_k0, ev_k1, ev_cnt;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    cudaEvent_t ev_dom0 = nullptr, ev_dom1 = nullptr;  // bracket the dominant kernel of a resident step
    float last_dom_ms = 0.f;
    // resident batch
    int res_n = 0;
    size_t res_bytes = 0;
    int res_fmt = -1;
    uint32_t res_tot[fg::K5_COUNT] = {};
    std::string last_error;
    int64_t launches = 0;
    int max_tile = 0;   // LTSV / GELF staging tile limit
    int max_tile5 = 0;  // RFC5424: tile + bitmap must fit the opt-in shared memory
};

namespace {

constexpr int kColW[9] = {8, 4, 8, 8, 8, 8, 8, 8, 8};  // ts(8) meta(4) host app proc msgid msg full sd (8 each)
enum { C_TS = 0, C_META, C_HOST, C_APP, C_PROC, C_MSGID, C_MSG, C_FULL, C_SD, C_COUNT };
size_t col_off(const fg_ctx* c, int col) {
    const size_t n = (size_t)c->max_lines;
    size_t o = 0;
    for (int k = 0; k < col; ++k) o += (size_t)kColW[k] * n;
    return o;
}

int fail(fg_ctx* c, int code, const char* what, cudaError_t e = cudaSuccess) {
    if (c) {
        c->last_error = what;
        if (e != cudaSuccess) {
            c->last_error += ": ";
            c->last_error += cudaGetErrorString(e);
        }
    }
    return code;
}

#define FG_CUDA(ctx, call)                                         \
    do {                                                           \
        cudaError_t _e = (call);                                   \
        if (_e != cudaSuccess) return fail(ctx, FG_E_CUDA, #call, _e); \
    } while (0)

template <class T>
void dfree(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}
template <class T>
void hfree(T*& p) {
    if (p) cudaFreeHost(p);
    p = nullptr;
}

uint32_t cap32(const Mirror& m) { return (uint32_t)std::min<size_t>(m.cap, 0xFFFFFFFFu); }

// The result tables of every format; capacities are in elements.  RFC3164 fills no side-table rows, but its results
// still point at an (empty) entries table.
void list_tables(fg_ctx* c) {
    const size_t mb = c->max_bytes;
    const std::vector<Mirror*> entries = {&c->entry_name, &c->entry_val, &c->entry_meta};
    c->tables[FG_FMT_RFC5424] = {{fg::K5_ENTRIES, {&c->e8}, std::max<size_t>(mb / 24, 4096), false},
                                 {fg::K5_ARENA, {&c->arena}, std::max<size_t>(mb / 64, 64 << 10), false},
                                 {fg::K5_WIDE_ROWS, {&c->wide}, 1024, false},
                                 {fg::K5_WIDE_ENTRIES, entries, 4096, false}};
    c->tables[FG_FMT_LTSV] = {{fg::K5_ENTRIES, entries, std::max<size_t>(mb / 24, 4096), true}};
    c->tables[FG_FMT_GELF] = c->tables[FG_FMT_LTSV];
    c->tables[FG_FMT_RFC3164] = {{fg::K5_ARENA, {&c->arena}, std::max<size_t>(mb / 32, 64 << 10), false},
                                 {fg::K5_ENTRIES, entries, 256, false}};
}

// Host arrays packed into one device allocation: every piece at a 16-byte aligned offset, 16 zero bytes after the last.
struct Blob {
    std::vector<uint8_t> bytes;
    template <class V>
    size_t put(const V& v) {  // a std::vector or std::string; returns its offset
        const size_t at = bytes.size();
        const uint8_t* p = (const uint8_t*)v.data();
        bytes.insert(bytes.end(), p, p + v.size() * sizeof(v[0]));
        bytes.resize((bytes.size() + 15) & ~(size_t)15, 0);
        return at;
    }
    cudaError_t upload(uint8_t*& d) {  // replaces d
        bytes.resize(bytes.size() + 16, 0);
        dfree(d);
        const cudaError_t e = cudaMalloc(&d, bytes.size());
        return e != cudaSuccess ? e : cudaMemcpy(d, bytes.data(), bytes.size(), cudaMemcpyHostToDevice);
    }
};

// packed zone table -> one device blob (fg::TzDeviceTable points into it)
int upload_tz(fg_ctx* c) {
    const fg::TzHostTable& H = c->tz_host;
    Blob b;
    const size_t o_hash = b.put(H.hash), o_key = b.put(H.key), o_zone = b.put(H.zone), o_noff = b.put(H.name_off),
                 o_first = b.put(H.first), o_off = b.put(H.off), o_names = b.put(H.names);
    FG_CUDA(c, b.upload(c->d_tz_blob));
    fg::TzDeviceTable& T = c->tz_dev;
    T = H.view();
    T.hash = (const unsigned long long*)(c->d_tz_blob + o_hash);
    T.key = (const long long*)(c->d_tz_blob + o_key);
    T.zone = (const int32_t*)(c->d_tz_blob + o_zone);
    T.name_off = (const int32_t*)(c->d_tz_blob + o_noff);
    T.first = (const int32_t*)(c->d_tz_blob + o_first);
    T.off = (const int32_t*)(c->d_tz_blob + o_off);
    T.names = c->d_tz_blob + o_names;
    return FG_OK;
}

// `OffsetDateTime::now_utc().year()` (rfc3164_decoder.rs:175): the configured year, else the clock's, once per call
int current_year(const fg_ctx* c) {
    if (c->r3164_year != 0) return c->r3164_year;
    const time_t now = time(nullptr);
    struct tm g;
    gmtime_r(&now, &g);
    return g.tm_year + 1900;
}

// Format-specific buffers are allocated on first use of the format.
int ensure_format(fg_ctx* c, int fmt) {
    if (fmt == FG_FMT_RFC5424 && !c->rows5.cap) {
        FG_CUDA(c, c->rows5.alloc(c->max_lines));
        FG_CUDA(c, cudaMalloc(&c->d_esc_list, (size_t)c->max_lines * 4));
    }
    if (fmt != FG_FMT_RFC5424 && !c->rows.cap) FG_CUDA(c, c->rows.alloc(col_off(c, C_COUNT)));
    if ((fmt == FG_FMT_RFC5424 || fmt == FG_FMT_GELF) && !c->d_wide_list)
        FG_CUDA(c, cudaMalloc(&c->d_wide_list, (size_t)c->max_lines * 4));
    for (const Table& t : c->tables[fmt]) {
        const size_t cap = t.cols[0]->cap;
        if (t.grow_to_first ? cap < t.first : cap == 0)
            for (Mirror* m : t.cols) FG_CUDA(c, m->alloc(t.first));
    }
    if (fmt == FG_FMT_RFC5424) return FG_OK;
    if (fmt == FG_FMT_RFC3164) {  // zone names need the database
        if (!c->tz_host.loaded) {
            std::string err;
            if (!fg::tz_load_dir(c->tzdir.empty() ? nullptr : c->tzdir.c_str(), c->tz_host, err)) return fail(c, FG_E_ARG, err.c_str());
        }
        if (!c->d_tz_blob)
            if (int rc = upload_tz(c)) return rc;
        return FG_OK;
    }
    // Scratch table for provisional side-table rows, indexed by byte offset (see Format<>::scratch_index):
    // a row needs >= 3 input bytes in GELF, >= 1 byte + its TAB in LTSV.
    const size_t need = (fmt == FG_FMT_LTSV ? c->max_bytes / 2 + (size_t)c->max_lines : c->max_bytes / 3) + 64;
    if (c->tmp_cap < need) {
        dfree(c->d_tmp_name); dfree(c->d_tmp_val); dfree(c->d_tmp_meta);
        c->tmp_cap = 0;
        FG_CUDA(c, cudaMalloc(&c->d_tmp_name, need * sizeof(int2)));
        FG_CUDA(c, cudaMalloc(&c->d_tmp_val, need * sizeof(unsigned long long)));
        FG_CUDA(c, cudaMalloc(&c->d_tmp_meta, need));
        c->tmp_cap = need;
    }
    return FG_OK;
}

// shared-memory tile: mean span of a CTA's lines plus slack; the kernel handles whatever does not fit in extra rounds
int pick_tile(const fg_ctx* c, size_t total_bytes, int n, int fmt) {
    const double mean = n > 0 ? (double)total_bytes / n : 0.0;
    const long lines = fg::lines_per_cta(fmt), gran = 8 * lines;  // 1 KiB steps for 128-line CTAs, 512 B for 64
#ifndef FG_TILE_SLACK_PCT  // head room of the tile over the mean span of a CTA's lines (profiles/variants.sh tries others)
#define FG_TILE_SLACK_PCT 102
#endif
    long t = (long)(mean * lines * (FG_TILE_SLACK_PCT / 100.0)) + gran;
    t = (t + gran - 1) / gran * gran;
    t = std::max(t, 8L * 1024);
    t = std::min(t, (long)(fmt == FG_FMT_RFC5424 ? c->max_tile5 : (fmt == FG_FMT_LTSV ? fg::kLtsvMaxTile : (fmt == FG_FMT_GELF ? fg::kGelfMaxTile : fg::kR3164MaxTile))));
    return (int)t;
}

// tables whose fill level the kernels report in the counter block
bool tables_overflow(const fg_ctx* c, int fmt, const uint32_t* t) {
    for (const Table& tb : c->tables[fmt])
        if (t[tb.slot] > tb.cols[0]->cap) return true;
    return false;
}
// the allocators kept counting past the capacity: grow each overflowed table once to the exact need
int regrow_tables(fg_ctx* c, int fmt, const uint32_t* t) {
    for (const Table& tb : c->tables[fmt]) {
        const size_t need = t[tb.slot];
        if (need > tb.cols[0]->cap)
            for (Mirror* m : tb.cols) FG_CUDA(c, m->alloc(need + need / 8 + 1024));
    }
    return FG_OK;
}

// One parse launch over lines [line0, line0 + n) of the resident offsets (for RFC5424: parse + unescape + wide kernels)
int launch_lines(fg_ctx* c, int fmt, int line0, int n, int tile, const uint8_t* invalid, int strip_eol, cudaStream_t s,
                 bool time_dominant = false) {
    if (fmt == FG_FMT_RFC5424) {
        fg::Parse5424Params P;
        P.bytes = c->d_bytes;
        P.offsets = c->offsets.dev<int32_t>() + line0;
        P.n = n;
        P.tile_bytes = tile;
        P.rows = c->rows5.dev<uint4>() + 2 * (size_t)line0;
        P.entries = c->e8.dev<unsigned long long>();
        P.entry_cap = cap32(c->e8);
        P.counters = c->d_k;
        P.esc_list = c->d_esc_list;
        P.wide_list = c->d_wide_list;
        P.arena = c->arena.d;
        P.arena_cap = cap32(c->arena);
        P.wide_rows = c->wide.dev<fg::WideRow>();
        P.wide_cap = cap32(c->wide);
        P.wentry_name = c->entry_name.dev<int2>();
        P.wentry_val = c->entry_val.dev<unsigned long long>();
        P.wentry_meta = c->entry_meta.d;
        P.wentry_cap = cap32(c->entry_name);
        P.line0 = line0;
        P.bad_offsets = c->d_k + fg::K5_BAD_OFFSETS;
        P.line_invalid = invalid;
        P.strip_eol = strip_eol;
        FG_CUDA(c, cudaMemsetAsync(c->d_k + fg::K5_ESC_LIST, 0, 8, s));  // the two work lists are per launch
        FG_CUDA(c, fg::launch_parse5424(P, s, time_dominant ? c->ev_dom0 : nullptr, time_dominant ? c->ev_dom1 : nullptr));
        c->launches += 2;  // parse5424_kernel + post5424_kernel
        return FG_OK;
    }
    fg::ParseParams P;
    P.bytes = c->d_bytes;
    P.offsets = c->offsets.dev<int32_t>() + line0;
    P.n = n;
    P.line0 = line0;
    P.tile_bytes = tile;
    uint8_t* r = c->rows.d;
    P.ts = (double*)(r + col_off(c, C_TS)) + line0;
    P.meta = (uint32_t*)(r + col_off(c, C_META)) + line0;
    P.host = (int2*)(r + col_off(c, C_HOST)) + line0;
    P.app = (int2*)(r + col_off(c, C_APP)) + line0;
    P.proc = (int2*)(r + col_off(c, C_PROC)) + line0;
    P.msgid = (int2*)(r + col_off(c, C_MSGID)) + line0;
    P.msg = (int2*)(r + col_off(c, C_MSG)) + line0;
    P.full = (int2*)(r + col_off(c, C_FULL)) + line0;
    P.sd = (int2*)(r + col_off(c, C_SD)) + line0;
    P.entry_name = c->entry_name.dev<int2>();
    P.entry_val = c->entry_val.dev<unsigned long long>();
    P.entry_meta = c->entry_meta.d;
    P.tmp_name = c->d_tmp_name;
    P.tmp_val = c->d_tmp_val;
    P.tmp_meta = c->d_tmp_meta;
    P.line_invalid = invalid;
    P.strip_eol = strip_eol;
    P.entry_counter = c->d_k + fg::K5_ENTRIES;
    P.entry_cap = cap32(c->entry_name);
    P.bad_offsets = c->d_k + fg::K5_BAD_OFFSETS;
    P.slow_list = c->d_wide_list;
    P.slow_count = c->d_k + fg::K5_WIDE_LIST;
    if (fmt == FG_FMT_GELF) FG_CUDA(c, cudaMemsetAsync(c->d_k + fg::K5_WIDE_LIST, 0, 4, s));  // the work list is per launch
    P.ltsv = c->ltsv;
    P.r3164.year = c->call_year;
    P.r3164.tz = c->tz_dev;
    P.r3164.arena = c->arena.d;
    P.r3164.arena_cap = cap32(c->arena);
    P.r3164.arena_counter = c->d_k + fg::K5_ARENA;
    if (time_dominant) FG_CUDA(c, cudaEventRecord(c->ev_dom0, s));
    FG_CUDA(c, fg::launch_parse(fmt, P, s));
    if (time_dominant) FG_CUDA(c, cudaEventRecord(c->ev_dom1, s));
    c->launches += fmt == FG_FMT_GELF ? 2 : 1;  // GELF: parse_gelf_kernel + post_gelf_kernel
    return FG_OK;
}

bool col_used(int col) { return !(col == C_APP || col == C_PROC || col == C_MSGID); }  // LTSV / GELF have no such fields

void fill_out(fg_ctx* c, int fmt, int n, const uint32_t* tot, fg_batch_out* out) {
    out->n = n;
    out->entry_name = c->entry_name.host<fg_span>();
    out->entry_val = c->entry_val.host<uint64_t>();
    out->entry_meta = c->entry_meta.h;
    if (fmt == FG_FMT_RFC5424) {
        out->n_entries = (int32_t)tot[fg::K5_WIDE_ENTRIES];
        out->rows5424 = c->rows5.host<fg_row5424>();
        out->entries8 = c->e8.host<uint64_t>();
        out->n_entries8 = (int32_t)tot[fg::K5_ENTRIES];
        out->n_wide = (int32_t)tot[fg::K5_WIDE_ROWS];
        out->wide_rows = c->wide.host<fg_wide_row>();
        out->arena = c->arena.h;
        out->arena_bytes = (int64_t)tot[fg::K5_ARENA];
        return;
    }
    uint8_t* r = c->rows.h;
    out->n_entries = (int32_t)tot[fg::K5_ENTRIES];
    if (fmt == FG_FMT_RFC3164) {
        out->n_entries = 0;
        out->arena = c->arena.h;
        out->arena_bytes = (int64_t)tot[fg::K5_ARENA];
    }
    out->ts = (const double*)(r + col_off(c, C_TS));
    out->meta = (const uint32_t*)(r + col_off(c, C_META));
    out->hostname = (const fg_span*)(r + col_off(c, C_HOST));
    out->msg = (const fg_span*)(r + col_off(c, C_MSG));
    out->full_msg = (const fg_span*)(r + col_off(c, C_FULL));
    out->sd = (const fg_span*)(r + col_off(c, C_SD));
}

int copy_rows_d2h(fg_ctx* c, int fmt, int line0, int n, cudaStream_t s) {
    if (n <= 0) return FG_OK;
    if (fmt == FG_FMT_RFC5424) {
        FG_CUDA(c, c->rows5.d2h(line0, line0 + n, s));
        return FG_OK;
    }
    // ts and meta: one copy each; the 8-byte span columns share one pitch (8 * max_lines), so every run of consecutive
    // used span columns goes back as ONE 2-D copy (few large D2H operations disturb the concurrent H2D stream less)
    for (int col = C_TS; col <= C_META; ++col) {
        const size_t o = col_off(c, col) + (size_t)line0 * kColW[col];
        FG_CUDA(c, c->rows.d2h(o, o + (size_t)n * kColW[col], s));
    }
    const size_t pitch = (size_t)c->max_lines * 8;
    int col = C_HOST;
    while (col < C_COUNT) {
        if (!col_used(col)) { ++col; continue; }
        int end = col;
        while (end + 1 < C_COUNT && col_used(end + 1)) ++end;
        const size_t o = col_off(c, col) + (size_t)line0 * 8;
        FG_CUDA(c, cudaMemcpy2DAsync(c->rows.h + o, pitch, c->rows.d + o, pitch, (size_t)n * 8, (size_t)(end - col + 1),
                                     cudaMemcpyDeviceToHost, s));
        col = end + 1;
    }
    return FG_OK;
}

// side tables on s_d2h: the rows a parse step produced are the contiguous range [prev, cur) of each bump allocator
int copy_tables_d2h(fg_ctx* c, int fmt, const uint32_t* prev, const uint32_t* cur) {
    for (const Table& tb : c->tables[fmt])
        for (const Mirror* m : tb.cols) FG_CUDA(c, m->d2h(prev[tb.slot], cur[tb.slot], c->s_d2h));
    return FG_OK;
}

bool is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// H2D of an arbitrary host range: direct DMA when pinned, else through two pinned bounce buffers
int h2d(fg_ctx* c, void* dst, const void* src, size_t bytes, bool pinned, int& bounce_ix) {
    if (!bytes) return FG_OK;
    if (pinned) {
        FG_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->s_h2d));
        return FG_OK;
    }
    size_t done = 0;
    while (done < bytes) {
        const size_t k = std::min(kBounceBytes, bytes - done);
        const int b = bounce_ix & 1;
        FG_CUDA(c, cudaEventSynchronize(c->bounce_ev[b]));
        memcpy(c->h_bounce[b], (const uint8_t*)src + done, k);
        FG_CUDA(c, cudaMemcpyAsync((uint8_t*)dst + done, c->h_bounce[b], k, cudaMemcpyHostToDevice, c->s_h2d));
        FG_CUDA(c, cudaEventRecord(c->bounce_ev[b], c->s_h2d));
        done += k;
        ++bounce_ix;
    }
    return FG_OK;
}

int ensure_events(fg_ctx* c, int chunks) {
    while ((int)c->ev_h2d.size() < chunks) {
        cudaEvent_t a, b, d, e;
        FG_CUDA(c, cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        FG_CUDA(c, cudaEventCreate(&b));
        FG_CUDA(c, cudaEventCreate(&d));
        FG_CUDA(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->ev_h2d.push_back(a);
        c->ev_k0.push_back(b);
        c->ev_k1.push_back(d);
        c->ev_cnt.push_back(e);
    }
    if (c->h_counts_cap < chunks) {
        hfree(c->h_counts);
        FG_CUDA(c, cudaHostAlloc(&c->h_counts, sizeof(uint32_t) * fg::K5_COUNT * (size_t)chunks, cudaHostAllocDefault));
        c->h_counts_cap = chunks;
    }
    return FG_OK;
}

// A caller's batch on its way to the device, chunk by chunk
struct Input {
    const uint8_t* bytes;
    const int32_t* offsets;
    bool pin_b, pin_o;
    int bounce_ix;
};

// Chunk k = lines [l0, l1) of a caller's batch: H2D of its bytes and offsets, then on s_comp the offsets check and,
// after ev_k0[k], the parse.
int enqueue_chunk(fg_ctx* c, int fmt, Input& in, int k, int l0, int l1, int tile) {
    const size_t b0 = (size_t)in.offsets[l0], b1 = (size_t)in.offsets[l1];
    if (b1 < b0 || b1 > c->max_bytes) {
        cudaDeviceSynchronize();
        return fail(c, FG_E_ARG, kBadOffsets);
    }
    int32_t* d_offsets = c->offsets.dev<int32_t>();
    if (int rc = h2d(c, c->d_bytes + b0, in.bytes + b0, b1 - b0, in.pin_b, in.bounce_ix)) return rc;
    if (int rc = h2d(c, d_offsets + l0, in.offsets + l0, sizeof(int32_t) * (size_t)(l1 - l0 + 1), in.pin_o, in.bounce_ix)) return rc;
    FG_CUDA(c, cudaEventRecord(c->ev_h2d[k], c->s_h2d));
    FG_CUDA(c, cudaStreamWaitEvent(c->s_comp, c->ev_h2d[k], 0));
    FG_CUDA(c, fg::launch_check_offsets(d_offsets + l0, l1 - l0, (long long)c->max_bytes, c->d_k + fg::K5_BAD_OFFSETS, c->s_comp));
    FG_CUDA(c, cudaEventRecord(c->ev_k0[k], c->s_comp));
    return launch_lines(c, fmt, l0, l1 - l0, tile, nullptr, 0, c->s_comp);
}

// Ends parse step j on stream s: ev_k1[j] closes its kernel time, the counter block is snapshotted into h_counts (with
// element j + 1 of `running`, if given), ev_cnt[j] marks the snapshot, and s_d2h waits for it before the step's
// results are copied back.
int end_step(fg_ctx* c, int j, cudaStream_t s, const Mirror* running = nullptr) {
    FG_CUDA(c, cudaEventRecord(c->ev_k1[j], s));
    FG_CUDA(c, cudaMemcpyAsync(c->h_counts + (size_t)j * fg::K5_COUNT, c->d_k, sizeof(uint32_t) * fg::K5_COUNT, cudaMemcpyDeviceToHost, s));
    if (running) FG_CUDA(c, running->d2h(j + 1, j + 2, s));
    FG_CUDA(c, cudaEventRecord(c->ev_cnt[j], s));
    FG_CUDA(c, cudaStreamWaitEvent(c->s_d2h, c->ev_cnt[j], 0));
    return FG_OK;
}

// Drains parse steps [0, steps) of one attempt, in order.  As soon as step j's counters arrive, `copy(j, prev, cur)`
// enqueues what step j produced on s_d2h while later steps are still in flight; it returns kRedo when a range of its
// own does not fit.  After an overflow nothing more is copied: the overflowed tables are grown to the exact need and
// kRedo asks the caller to enqueue the attempt again.  Otherwise *kms is the summed kernel time of the steps.
// total receives the last snapshot.
template <class Copy>
int drain(fg_ctx* c, int fmt, int steps, Copy&& copy, uint32_t* total, float* kms) {
    uint32_t prev[fg::K5_COUNT] = {};
    memset(total, 0, sizeof prev);
    bool overflow = false;
    for (int j = 0; j < steps; ++j) {
        FG_CUDA(c, cudaEventSynchronize(c->ev_cnt[j]));
        const uint32_t* cur = c->h_counts + (size_t)j * fg::K5_COUNT;
        memcpy(total, cur, sizeof prev);
        overflow = overflow || tables_overflow(c, fmt, cur);
        if (overflow) continue;  // keep draining the events; the attempt is redone below
        const int rc = copy(j, prev, cur);
        if (rc == kRedo) overflow = true;
        else if (rc) return rc;
        memcpy(prev, cur, sizeof prev);
    }
    FG_CUDA(c, cudaStreamSynchronize(c->s_d2h));
    if (total[fg::K5_BAD_OFFSETS]) return fail(c, FG_E_ARG, kBadOffsets);
    if (overflow) {
        if (int rc = regrow_tables(c, fmt, total)) return rc;
        return kRedo;
    }
    *kms = 0.f;
    for (int j = 0; j < steps; ++j) {
        float ms = 0.f;
        FG_CUDA(c, cudaEventElapsedTime(&ms, c->ev_k0[j], c->ev_k1[j]));
        *kms += ms;
    }
    return FG_OK;
}

// Cheap host-side checks; the interior of the offsets array is checked on the device (check_offsets_kernel) next to
// the parse, so a non-monotone or out-of-range offset fails the call with FG_E_ARG instead of reaching a kernel.
int check_batch(fg_ctx* c, const uint8_t* bytes, const int32_t* offsets, int32_t n) {
    if (!c) return FG_E_ARG;
    if (n < 0 || (n > 0 && (!bytes || !offsets))) return fail(c, FG_E_ARG, "null input");
    if (n > c->max_lines) return fail(c, FG_E_CAPACITY, "batch has more lines than max_batch_lines");
    if (n > 0) {
        if (offsets[0] < 0 || offsets[n] < offsets[0]) return fail(c, FG_E_ARG, "offsets must be non-negative and non-decreasing");
        if ((size_t)offsets[n] > c->max_bytes) return fail(c, FG_E_CAPACITY, "batch has more bytes than max_batch_bytes");
    }
    return FG_OK;
}

// serde_json 0.8 escape_bytes, for the keys / values of output.gelf_extra rendered once on the host
void json_escape_into(const std::string& v, std::string& o) {
    o.push_back('"');
    for (const char c : v) {
        switch (c) {
            case '"': o += "\\\""; break;
            case '\\': o += "\\\\"; break;
            case '\x08': o += "\\b"; break;
            case '\x0c': o += "\\f"; break;
            case '\n': o += "\\n"; break;
            case '\r': o += "\\r"; break;
            case '\t': o += "\\t"; break;
            default: o.push_back(c);
        }
    }
    o.push_back('"');
}

// The keys GelfEncoder::encode always or conditionally inserts (gelf_encoder.rs:60-100) merged with output.gelf_extra
// (:110-112, inserted last: an extra replaces a fixed key of the same name), sorted by key like the BTreeMap iterates.
int build_static_items(fg_ctx* c) {
    struct Item { std::string key, lit; int kind; };
    static const char* fixed[9] = {"application_name", "full_message", "host", "level", "process_id", "sd_id", "short_message",
                                   "timestamp", "version"};
    std::vector<Item> items;
    for (int k = 0; k < 9; ++k) {
        Item it;
        it.key = fixed[k];
        it.lit = ",";  // the device skips the comma for the first item of a record
        json_escape_into(it.key, it.lit);
        it.lit.push_back(':');
        it.kind = k;
        items.push_back(it);
    }
    for (const auto& kv : c->gelf_extra) {
        Item it;
        it.key = kv.first;
        it.lit = ",";
        json_escape_into(kv.first, it.lit);
        it.lit.push_back(':');
        json_escape_into(kv.second, it.lit);
        it.kind = 100;
        bool replaced = false;
        for (auto& x : items)
            if (x.key == it.key) { x = it; replaced = true; }
        if (!replaced) items.push_back(it);
    }
    std::sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.key < b.key; });  // byte order (std::string compares as unsigned char)
    std::vector<int32_t> key_off{0}, lit_off, kind;
    std::string blob;
    for (const auto& it : items) {
        blob += it.key;
        key_off.push_back((int32_t)blob.size());
    }
    lit_off.push_back((int32_t)blob.size());
    for (const auto& it : items) {
        blob += it.lit;
        lit_off.push_back((int32_t)blob.size());
        kind.push_back(it.kind);
    }
    Blob b;
    b.put(blob);  // at offset 0: d_static_blob is the base of key_off / lit_off
    const size_t o_key = b.put(key_off), o_lit = b.put(lit_off), o_kind = b.put(kind);
    FG_CUDA(c, b.upload(c->d_static_blob));
    c->n_static = (int)items.size();
    c->d_static_key_off = (const int32_t*)(c->d_static_blob + o_key);
    c->d_static_lit_off = (const int32_t*)(c->d_static_blob + o_lit);
    c->d_static_kind = (const int32_t*)(c->d_static_blob + o_kind);
    return FG_OK;
}

int ensure_encoder(fg_ctx* c, int chunks) {
    if (!c->d_enc_lens) {
        FG_CUDA(c, cudaMalloc(&c->d_enc_lens, (size_t)c->max_lines * 4));
        FG_CUDA(c, cudaMalloc(&c->d_enc_rel, (size_t)c->max_lines * 4));
        FG_CUDA(c, c->enc_offsets.alloc((size_t)c->max_lines + 1));
        FG_CUDA(c, c->enc_status.alloc(c->max_lines));
        c->scan_temp_bytes = fg::gelf_scan_temp_bytes(c->max_lines);
        FG_CUDA(c, cudaMalloc(&c->d_scan_temp, c->scan_temp_bytes + 256));
    }
    if (!c->enc_out.cap) FG_CUDA(c, c->enc_out.alloc(c->max_bytes * 2 + (size_t)c->max_lines * 200));
    if (c->enc_base.cap < (size_t)chunks + 1) FG_CUDA(c, c->enc_base.alloc((size_t)chunks + 1));
    if (!c->d_static_blob)
        if (int rc = build_static_items(c)) return rc;
    return FG_OK;
}

}  // namespace

extern "C" {

int fg_create(const fg_config* cfg, fg_ctx** out) {
    if (!out) return FG_E_ARG;
    *out = nullptr;
    fg_config def{};
    if (!cfg) cfg = &def;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return FG_E_NO_DEVICE;  // no CPU fallback: the decoder does not exist without a GPU
    }
    if (cfg->device < 0 || cfg->device >= ndev) return FG_E_ARG;
    fg_ctx* c = new (std::nothrow) fg_ctx();
    if (!c) return FG_E_ARG;
    c->device = cfg->device;
    c->max_bytes = cfg->max_batch_bytes > 0 ? (size_t)cfg->max_batch_bytes : ((size_t)256 << 20);
    if (c->max_bytes > 0x7FFFFFC0ull) c->max_bytes = 0x7FFFFFC0ull;  // int32 offsets
    c->max_lines = cfg->max_batch_lines > 0 ? cfg->max_batch_lines : (2 << 20);
    c->max_lines = (c->max_lines + 63) & ~63;  // keeps every row column 256-byte aligned
    c->chunk_lines = cfg->chunk_lines > 0 ? cfg->chunk_lines : (512 << 10);  // measured: 246 / 258 / 258 M lines/s e2e at 128 Ki / 512 Ki / 1 Mi lines per chunk (profiles/r2_notes.md)
    c->chunk_lines = (c->chunk_lines + 127) / 128 * 128;  // a multiple of every kernel's lines per CTA
    c->r3164_year = cfg->rfc3164_year;
    if (cfg->tzdir) c->tzdir = cfg->tzdir;
    list_tables(c);
#define FG_CREATE_CUDA(call)                                 \
    do {                                                      \
        cudaError_t _e = (call);                              \
        if (_e != cudaSuccess) {                              \
            fprintf(stderr, "flowgger_cuda: %s failed: %s\n", #call, cudaGetErrorString(_e)); \
            fg_destroy(c);                                    \
            return FG_E_CUDA;                                 \
        }                                                     \
    } while (0)
    FG_CREATE_CUDA(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    FG_CREATE_CUDA(cudaGetDeviceProperties(&prop, c->device));
    c->max_tile = (int)std::min<size_t>(prop.sharedMemPerBlockOptin - 1024, 200 * 1024);
    c->max_tile &= ~1023;
    c->max_tile5 = (int)(((size_t)c->max_tile - 1024) * 8 / 9) & ~1023;  // tile + tile/8 bitmap + static shared memory
    FG_CREATE_CUDA(fg::configure_kernels(c->max_tile, c->max_tile5));
    FG_CREATE_CUDA(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
    FG_CREATE_CUDA(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
    FG_CREATE_CUDA(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
    FG_CREATE_CUDA(cudaEventCreate(&c->ev_a));
    FG_CREATE_CUDA(cudaEventCreate(&c->ev_b));
    FG_CREATE_CUDA(cudaEventCreate(&c->ev_dom0));
    FG_CREATE_CUDA(cudaEventCreate(&c->ev_dom1));
    FG_CREATE_CUDA(cudaMalloc(&c->d_bytes, c->max_bytes + kPad));
    FG_CREATE_CUDA(cudaMemset(c->d_bytes + c->max_bytes, 0, kPad));
    FG_CREATE_CUDA(c->offsets.alloc((size_t)c->max_lines + 1));
    FG_CREATE_CUDA(cudaMalloc(&c->d_k, 256));
    FG_CREATE_CUDA(cudaMemset(c->d_k, 0, 256));
    for (int b = 0; b < 2; ++b) {
        FG_CREATE_CUDA(cudaHostAlloc(&c->h_bounce[b], kBounceBytes, cudaHostAllocDefault));
        FG_CREATE_CUDA(cudaEventCreateWithFlags(&c->bounce_ev[b], cudaEventDisableTiming));
    }
    // LTSV schema / suffixes -> one device blob
    {
        std::vector<uint8_t> names, suffix;
        std::vector<int32_t> name_off{0}, types;
        const int ns = (cfg->ltsv_schema_names && cfg->ltsv_schema_types) ? cfg->ltsv_schema_len : 0;
        for (int k = 0; k < ns; ++k) {
            const char* s = cfg->ltsv_schema_names[k];
            names.insert(names.end(), (const uint8_t*)s, (const uint8_t*)s + strlen(s));
            name_off.push_back((int32_t)names.size());
            types.push_back(cfg->ltsv_schema_types[k]);
        }
        fg::LtsvDeviceConfig& L = c->ltsv;
        L.has_schema = (cfg->ltsv_has_schema || ns > 0) ? 1 : 0;
        L.n_schema = ns;
        L.suffix_present = 0;
        L.suffix_off[0] = 0;
        for (int t = 0; t < 5; ++t) {
            const char* s = cfg->ltsv_suffix[t];
            if (t > 0 && s) {
                L.suffix_present |= 1u << t;
                suffix.insert(suffix.end(), (const uint8_t*)s, (const uint8_t*)s + strlen(s));
            }
            L.suffix_off[t + 1] = (int32_t)suffix.size();
        }
        Blob b;
        const size_t o_names = b.put(names), o_off = b.put(name_off), o_types = b.put(types), o_suf = b.put(suffix);
        FG_CREATE_CUDA(b.upload(c->d_ltsv_blob));
        L.names = c->d_ltsv_blob + o_names;
        L.name_off = (const int32_t*)(c->d_ltsv_blob + o_off);
        L.types = (const int32_t*)(c->d_ltsv_blob + o_types);
        L.suffix = c->d_ltsv_blob + o_suf;
    }
#undef FG_CREATE_CUDA
    *out = c;
    return FG_OK;
}

void fg_destroy(fg_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    dfree(c->d_bytes); dfree(c->d_k); dfree(c->d_flush); dfree(c->d_esc_list); dfree(c->d_wide_list);
    dfree(c->d_enc_lens); dfree(c->d_enc_rel); dfree(c->d_scan_temp);
    dfree(c->d_static_blob);
    dfree(c->d_seg); dfree(c->d_n_lines); dfree(c->d_invalid);
    hfree(c->h_n_lines);
    if (c->s_parse) cudaStreamDestroy(c->s_parse);
    for (auto e : c->ev_split) cudaEventDestroy(e);
    if (c->ev_s0) cudaEventDestroy(c->ev_s0);
    if (c->ev_s1) cudaEventDestroy(c->ev_s1);
    dfree(c->d_tmp_name); dfree(c->d_tmp_val); dfree(c->d_tmp_meta);
    dfree(c->d_ltsv_blob);
    dfree(c->d_tz_blob);
    hfree(c->h_counts);
    for (int b = 0; b < 2; ++b) {
        hfree(c->h_bounce[b]);
        if (c->bounce_ev[b]) cudaEventDestroy(c->bounce_ev[b]);
    }
    for (auto e : c->ev_h2d) cudaEventDestroy(e);
    for (auto e : c->ev_k0) cudaEventDestroy(e);
    for (auto e : c->ev_k1) cudaEventDestroy(e);
    for (auto e : c->ev_cnt) cudaEventDestroy(e);
    if (c->ev_a) cudaEventDestroy(c->ev_a);
    if (c->ev_b) cudaEventDestroy(c->ev_b);
    if (c->ev_dom0) cudaEventDestroy(c->ev_dom0);
    if (c->ev_dom1) cudaEventDestroy(c->ev_dom1);
    if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
    if (c->s_comp) cudaStreamDestroy(c->s_comp);
    if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
    delete c;  // the mirrors release themselves
}

const char* fg_last_error(const fg_ctx* c) { return c ? c->last_error.c_str() : "null context"; }

int fg_host_alloc(fg_ctx* c, size_t bytes, void** out) {
    if (!c || !out) return FG_E_ARG;
    FG_CUDA(c, cudaSetDevice(c->device));
    FG_CUDA(c, cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return FG_OK;
}
void fg_host_free(fg_ctx* c, void* p) {
    if (c && p) cudaFreeHost(p);
}

int fg_decode_batch(fg_ctx* c, fg_format fmt, const uint8_t* bytes, const int32_t* offsets, int32_t n,
                    fg_batch_out* out) {
    if (!c || !out) return FG_E_ARG;
    if (int rc = check_batch(c, bytes, offsets, n)) return rc;
    if ((int)fmt < 0 || (int)fmt > 3) return fail(c, FG_E_ARG, "unknown format");
    FG_CUDA(c, cudaSetDevice(c->device));
    if (int rc = ensure_format(c, (int)fmt)) return rc;
    c->call_year = current_year(c);
    memset(out, 0, sizeof *out);
    const uint32_t zero[fg::K5_COUNT] = {};
    if (n == 0) {
        fill_out(c, fmt, 0, zero, out);
        return FG_OK;
    }
    const auto t_begin = std::chrono::steady_clock::now();
    Input in{bytes, offsets, is_pinned(bytes), is_pinned(offsets), 0};
    const int C = c->chunk_lines;
    const int chunks = (n + C - 1) / C;
    if (int rc = ensure_events(c, chunks)) return rc;
    const int tile = pick_tile(c, (size_t)(offsets[n] - offsets[0]), n, (int)fmt);
    auto copy_tables = [&](int, const uint32_t* prev, const uint32_t* cur) { return copy_tables_d2h(c, fmt, prev, cur); };
    for (int attempt = 0; attempt < 2; ++attempt) {
        FG_CUDA(c, cudaMemsetAsync(c->d_k, 0, sizeof(uint32_t) * fg::K5_COUNT, c->s_comp));
        in.bounce_ix = 0;
        for (int k = 0; k < chunks; ++k) {
            const int l0 = k * C, l1 = std::min(n, l0 + C);
            if (int rc = enqueue_chunk(c, fmt, in, k, l0, l1, tile)) return rc;
            if (int rc = end_step(c, k, c->s_comp)) return rc;
            if (int rc = copy_rows_d2h(c, fmt, l0, l1 - l0, c->s_d2h)) return rc;
        }
        uint32_t total[fg::K5_COUNT];
        float kms = 0.f;
        const int rc = drain(c, fmt, chunks, copy_tables, total, &kms);
        if (rc == kRedo) continue;
        if (rc) return rc;
        fill_out(c, fmt, n, total, out);
        out->kernel_ms = kms;
        out->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        return FG_OK;
    }
    return fail(c, FG_E_CAPACITY, "side table overflow after regrow");
}

int fg_set_rfc3164_year(fg_ctx* c, int32_t year) {
    if (!c) return FG_E_ARG;
    c->r3164_year = year;
    return FG_OK;
}

int fg_set_tz_table(fg_ctx* c, int32_t n_zones, const char* const* names, const int32_t* first, const int64_t* span_start_utc,
                    const int32_t* span_offset) {
    if (!c || n_zones < 0 || (n_zones > 0 && (!names || !first || !span_start_utc || !span_offset))) return FG_E_ARG;
    std::vector<std::string> nm;
    std::vector<fg::TzZoneSpans> zones;
    if (n_zones > 0 && first[0] < 0) return fail(c, FG_E_ARG, "fg_set_tz_table: first[] must start at a non-negative index");
    for (int32_t z = 0; z < n_zones; ++z) {
        const int32_t a = first[z], b = first[z + 1];
        if (!names[z] || !names[z][0] || b <= a) return fail(c, FG_E_ARG, "fg_set_tz_table: every zone needs a name and at least one span");
        fg::TzZoneSpans sp;
        for (int32_t j = a; j < b; ++j) {
            if (j > a) {
                if (j > a + 1 && span_start_utc[j] <= span_start_utc[j - 1]) return fail(c, FG_E_ARG, "fg_set_tz_table: span starts must ascend");
                sp.trans.push_back((long long)span_start_utc[j]);
            }
            sp.offs.push_back(span_offset[j]);
        }
        nm.emplace_back(names[z]);
        zones.push_back(std::move(sp));
    }
    FG_CUDA(c, cudaSetDevice(c->device));
    FG_CUDA(c, cudaDeviceSynchronize());
    fg::tz_build(nm, zones, c->tz_host);
    return upload_tz(c);
}

// host-side queries of the zone database (no device involved), for callers that want to check what a context will load
namespace {
std::mutex g_tz_mu;
std::string g_tz_dir;
fg::TzHostTable g_tz_table;
bool tz_query_table(const char* tzdir) {  // g_tz_mu held
    const std::string dir = tzdir ? tzdir : "";
    if (g_tz_table.loaded && dir == g_tz_dir) return true;
    std::string err;
    fg::TzHostTable t;
    if (!fg::tz_load_dir(tzdir, t, err)) return false;
    g_tz_table = std::move(t);
    g_tz_dir = dir;
    return true;
}
}  // namespace

// what get_by_name + assume_timezone answer for `name` at the local second `local`:
// 1 = found (offset stored), 0 = no such identifier, FG_E_ARG = the database could not be read
int fg_tz_lookup(const char* tzdir, const char* name, int64_t local, int32_t* offset) {
    if (!name) return FG_E_ARG;
    std::lock_guard<std::mutex> guard(g_tz_mu);
    if (!tz_query_table(tzdir)) return FG_E_ARG;
    const fg::TzDeviceTable T = g_tz_table.view();
    const int z = fg::tz_find(T, (const uint8_t*)name, 0, (int)strlen(name));
    if (z < 0) return 0;
    if (offset) *offset = fg::tz_offset_local(T, z, (long long)local);
    return 1;
}
// identifiers in the database under `tzdir` (negative: unreadable)
int32_t fg_tz_count(const char* tzdir) {
    std::lock_guard<std::mutex> guard(g_tz_mu);
    if (!tz_query_table(tzdir)) return FG_E_ARG;
    return (int32_t)g_tz_table.n_names();
}

int fg_set_gelf_extra(fg_ctx* c, int32_t n, const char* const* keys, const char* const* values) {
    if (!c || n < 0 || (n > 0 && (!keys || !values))) return FG_E_ARG;
    FG_CUDA(c, cudaSetDevice(c->device));
    c->gelf_extra.clear();
    for (int32_t k = 0; k < n; ++k) {
        if (!keys[k] || !values[k]) return fail(c, FG_E_ARG, "output.gelf_extra values must be strings");  // gelf_encoder.rs:41
        c->gelf_extra.emplace_back(keys[k], values[k]);
    }
    FG_CUDA(c, cudaDeviceSynchronize());
    return build_static_items(c);
}

// decode (RFC5424) + GelfEncoder::encode fused: H2D lines -> parse kernels -> size / scan / write kernels -> D2H of the
// encoded records only, chunk by chunk; the decoder's rows and side tables never leave the device.
int fg_decode_encode_gelf(fg_ctx* c, fg_format fmt, const uint8_t* bytes, const int32_t* offsets, int32_t n, fg_encoded_out* out) {
    if (!c || !out) return FG_E_ARG;
    if (int rc = check_batch(c, bytes, offsets, n)) return rc;
    if (fmt != FG_FMT_RFC5424) return fail(c, FG_E_ARG, "the fused encoder takes input.format = rfc5424");
    FG_CUDA(c, cudaSetDevice(c->device));
    if (int rc = ensure_format(c, (int)fmt)) return rc;
    c->call_year = current_year(c);
    const int C = c->chunk_lines;
    const int chunks = n > 0 ? (n + C - 1) / C : 1;
    if (int rc = ensure_encoder(c, chunks)) return rc;
    memset(out, 0, sizeof *out);
    out->bytes = c->enc_out.h;
    out->offsets = c->enc_offsets.host<int64_t>();
    out->status = c->enc_status.h;
    if (n == 0) {
        c->enc_offsets.host<int64_t>()[0] = 0;
        return FG_OK;
    }
    const auto t_begin = std::chrono::steady_clock::now();
    Input in{bytes, offsets, is_pinned(bytes), is_pinned(offsets), 0};
    if (int rc = ensure_events(c, chunks)) return rc;
    const int tile = pick_tile(c, (size_t)(offsets[n] - offsets[0]), n, (int)fmt);
    // encoded bytes: chunk k's records are the contiguous range [base(k), base(k+1)) of the output
    unsigned long long* base = c->enc_base.host<unsigned long long>();
    base[0] = 0;
    auto copy_records = [&](int k, const uint32_t*, const uint32_t*) {
        if (base[k + 1] > c->enc_out.cap) return kRedo;
        FG_CUDA(c, c->enc_out.d2h(base[k], base[k + 1], c->s_d2h));
        return FG_OK;
    };
    for (int attempt = 0; attempt < 3; ++attempt) {
        FG_CUDA(c, cudaMemsetAsync(c->d_k, 0, sizeof(uint32_t) * fg::K5_COUNT, c->s_comp));
        FG_CUDA(c, cudaMemsetAsync(c->enc_base.d, 0, sizeof(unsigned long long), c->s_comp));
        in.bounce_ix = 0;
        for (int k = 0; k < chunks; ++k) {
            const int l0 = k * C, l1 = std::min(n, l0 + C);
            if (int rc = enqueue_chunk(c, fmt, in, k, l0, l1, tile)) return rc;
            fg::GelfEncodeParams E;
            E.bytes = c->d_bytes;
            E.offsets = c->offsets.dev<int32_t>() + l0;
            E.n = l1 - l0;
            E.rows = c->rows5.dev<uint4>() + 2 * (size_t)l0;
            E.entries = c->e8.dev<unsigned long long>();
            E.arena = c->arena.d;
            E.wide_rows = c->wide.dev<fg::WideRow>();
            E.wentry_name = c->entry_name.dev<int2>();
            E.wentry_val = c->entry_val.dev<unsigned long long>();
            E.wentry_meta = c->entry_meta.d;
            E.static_blob = c->d_static_blob;
            E.n_static = c->n_static;
            E.static_key_off = c->d_static_key_off;
            E.static_lit_off = c->d_static_lit_off;
            E.static_kind = c->d_static_kind;
            E.lens = c->d_enc_lens + l0;
            E.rel = c->d_enc_rel + l0;
            E.base = c->enc_base.dev<unsigned long long>() + k;
            E.out = c->enc_out.d;
            E.out_cap = c->enc_out.cap;
            E.out_offsets = c->enc_offsets.dev<long long>() + l0;
            E.status = c->enc_status.d + l0;
            E.bad_offsets = c->d_k + fg::K5_BAD_OFFSETS;
            E.entry_cap = cap32(c->e8);
            E.wide_cap = cap32(c->wide);
            E.wentry_cap = cap32(c->entry_name);
            E.tile_bytes = std::min(4 * tile, c->max_tile5);  // the encoder's CTAs take 256 lines (4 x the parse kernel's 64)
            FG_CUDA(c, fg::launch_gelf_encode(E, c->d_scan_temp, c->scan_temp_bytes, c->s_comp));
            c->launches += 4;
            if (int rc = end_step(c, k, c->s_comp, &c->enc_base)) return rc;
            FG_CUDA(c, c->enc_status.d2h(l0, l1, c->s_d2h));
            FG_CUDA(c, c->enc_offsets.d2h(l0, l1 + 1, c->s_d2h));
        }
        uint32_t total[fg::K5_COUNT];
        float kms = 0.f;
        const int rc = drain(c, fmt, chunks, copy_records, total, &kms);
        if (rc == kRedo) {
            const unsigned long long need = base[chunks];
            if (need > c->enc_out.cap) FG_CUDA(c, c->enc_out.alloc((size_t)need + (size_t)need / 8 + 4096));
            out->bytes = c->enc_out.h;
            continue;
        }
        if (rc) return rc;
        out->n = n;
        out->kernel_ms = kms;
        out->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        return FG_OK;
    }
    return fail(c, FG_E_CAPACITY, "output / side table overflow after regrow");
}

int fg_split_decode(fg_ctx* c, fg_format fmt, const uint8_t* stream, int64_t nbytes, fg_batch_out* out) {
    return fg_split_decode_framed(c, fmt, FG_FRAME_LINE, stream, nbytes, out);
}

int fg_split_decode_framed(fg_ctx* c, fg_format fmt, fg_framing framing, const uint8_t* stream, int64_t nbytes, fg_batch_out* out) {
    if (!c || !out) return FG_E_ARG;
    if ((int)fmt < 0 || (int)fmt > 3) return fail(c, FG_E_ARG, "unknown format");
    if (framing != FG_FRAME_LINE && framing != FG_FRAME_NUL) return fail(c, FG_E_ARG, "unknown framing");
    const int delim = framing == FG_FRAME_NUL ? 0 : '\n';
    const int strip = framing == FG_FRAME_NUL ? 2 : 1;
    if (nbytes < 0 || (nbytes > 0 && !stream)) return fail(c, FG_E_ARG, "null input");
    if ((size_t)nbytes > c->max_bytes) return fail(c, FG_E_CAPACITY, "stream has more bytes than max_batch_bytes");
    FG_CUDA(c, cudaSetDevice(c->device));
    if (int rc = ensure_format(c, (int)fmt)) return rc;
    c->call_year = current_year(c);
    const auto t_begin = std::chrono::steady_clock::now();
    constexpr long long kChunk = 64ll << 20;  // pipeline granularity in bytes (a multiple of the 8 KB framing segment)
    const int chunks = nbytes > 0 ? (int)((nbytes + kChunk - 1) / kChunk) : 1;
    if (!c->d_seg) {
        FG_CUDA(c, cudaMalloc(&c->d_seg, sizeof(uint32_t) * ((size_t)fg::split_segments((long long)c->max_bytes) + 16)));
        FG_CUDA(c, cudaMalloc(&c->d_n_lines, 256));
        FG_CUDA(c, cudaMalloc(&c->d_invalid, (size_t)c->max_lines + 64));
        FG_CUDA(c, cudaHostAlloc(&c->h_n_lines, 64, cudaHostAllocDefault));
        FG_CUDA(c, cudaEventCreate(&c->ev_s0));
        FG_CUDA(c, cudaEventCreate(&c->ev_s1));
        FG_CUDA(c, cudaStreamCreateWithFlags(&c->s_parse, cudaStreamNonBlocking));
    }
    if ((int)c->ev_split.size() < chunks + 1) {
        const size_t want = (size_t)chunks + 1;
        while (c->ev_split.size() < want) {
            cudaEvent_t e;
            FG_CUDA(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            c->ev_split.push_back(e);
        }
        FG_CUDA(c, c->cum.alloc(want));
    }
    if (int rc = ensure_events(c, chunks + 1)) return rc;
    memset(out, 0, sizeof *out);
    const bool pinned = nbytes > 0 && is_pinned(stream);
    const int32_t* cum = c->cum.host<int32_t>();
    auto copy_tables = [&](int, const uint32_t* prev, const uint32_t* cur) { return copy_tables_d2h(c, fmt, prev, cur); };

    for (int attempt = 0; attempt < 2; ++attempt) {
        // ---- enqueue, chunk by chunk: raw bytes -> HBM, then framing + UTF-8 validation of that chunk (no host dependency)
        FG_CUDA(c, cudaMemsetAsync(c->d_n_lines + 8, 0, 4, c->s_comp));  // running newline count (uint32 at d_n_lines[8])
        FG_CUDA(c, cudaMemsetAsync(c->d_invalid, 0, (size_t)c->max_lines, c->s_comp));
        FG_CUDA(c, cudaMemsetAsync(c->d_k, 0, sizeof(uint32_t) * fg::K5_COUNT, c->s_comp));
        FG_CUDA(c, cudaEventRecord(c->ev_s0, c->s_comp));
        int bounce_ix = 0;
        for (int k = 0; k < chunks; ++k) {
            const long long c0 = (long long)k * kChunk, c1 = std::min<long long>(nbytes, c0 + kChunk);
            const bool last = k == chunks - 1;
            if (int rc = h2d(c, c->d_bytes + c0, stream + c0, (size_t)(c1 - c0), pinned, bounce_ix)) return rc;
            if (last) FG_CUDA(c, cudaMemsetAsync(c->d_bytes + nbytes, delim ? 0 : 0xFF, 64, c->s_h2d));  // whole-vector loads past the end see no delimiter
            FG_CUDA(c, cudaEventRecord(c->ev_h2d[k], c->s_h2d));
            FG_CUDA(c, cudaStreamWaitEvent(c->s_comp, c->ev_h2d[k], 0));
            FG_CUDA(c, fg::launch_split_chunk(c->d_bytes, (long long)nbytes, c0, c1, last ? 1 : 0, c->d_seg, (uint32_t*)(c->d_n_lines + 8),
                                              c->cum.dev<int32_t>() + k, c->offsets.dev<int32_t>(), c->d_n_lines, c->max_lines,
                                              c->d_invalid, delim, c->s_comp));
            c->launches += 4;
            FG_CUDA(c, c->cum.d2h(k, k + 1, c->s_comp));
            if (last) {
                FG_CUDA(c, cudaMemcpyAsync(c->h_n_lines, c->d_n_lines, 4, cudaMemcpyDeviceToHost, c->s_comp));
                FG_CUDA(c, cudaEventRecord(c->ev_s1, c->s_comp));
            }
            FG_CUDA(c, cudaEventRecord(c->ev_split[k], c->s_comp));
        }
        // ---- parse the lines that END in chunk k once chunk k+1 has been validated too (a sequence that starts in the
        //      last 16 bytes of a chunk is checked with the next one); rows go back while later chunks are still in flight
        int32_t done_lines = 0;
        int32_t n = 0;
        int nparse = 0;
        bool over = false;
        for (int k = 0; k < chunks; ++k) {
            const int dep = std::min(k + 1, chunks - 1);
            FG_CUDA(c, cudaEventSynchronize(c->ev_split[dep]));
            int32_t upto = cum[k];
            if (upto < 0) { over = true; break; }
            if (k == chunks - 1) {
                n = *c->h_n_lines;
                if (n < 0) { over = true; break; }
                upto = n;  // includes an unterminated last line
            }
            const int32_t cnt = upto - done_lines;
            if (cnt > 0) {
                const size_t span_bytes = (size_t)std::min<long long>(nbytes, (long long)(k + 1) * kChunk) - (size_t)((long long)k * kChunk);
                const int tile = pick_tile(c, std::max<size_t>(span_bytes, 1), cnt, (int)fmt);
                FG_CUDA(c, cudaStreamWaitEvent(c->s_parse, c->ev_split[dep], 0));
                FG_CUDA(c, cudaEventRecord(c->ev_k0[nparse], c->s_parse));
                if (int rc = launch_lines(c, (int)fmt, done_lines, cnt, tile, c->d_invalid + done_lines, strip, c->s_parse)) return rc;
                if (int rc = end_step(c, nparse, c->s_parse)) return rc;
                if (int rc = copy_rows_d2h(c, fmt, done_lines, cnt, c->s_d2h)) return rc;
                ++nparse;
                done_lines = upto;
            }
        }
        if (over) {
            FG_CUDA(c, cudaDeviceSynchronize());
            return fail(c, FG_E_CAPACITY, "stream has more lines than max_batch_lines");
        }
        // ---- side table ranges, line offsets
        uint32_t total[fg::K5_COUNT];
        float kms = 0.f;
        const int rc = drain(c, fmt, nparse, copy_tables, total, &kms);
        if (rc == kRedo) continue;
        if (rc) return rc;
        FG_CUDA(c, cudaStreamSynchronize(c->s_parse));
        FG_CUDA(c, c->offsets.d2h(0, (size_t)n + 1, c->s_d2h));
        FG_CUDA(c, cudaStreamSynchronize(c->s_d2h));
        FG_CUDA(c, cudaEventElapsedTime(&c->last_split_ms, c->ev_s0, c->ev_s1));  // includes waiting for the H2D chunks
        fill_out(c, fmt, n, total, out);
        out->line_offsets = c->offsets.host<int32_t>();
        out->kernel_ms = kms;
        out->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        return FG_OK;
    }
    return fail(c, FG_E_CAPACITY, "side table overflow after regrow");
}

int fg_upload(fg_ctx* c, const uint8_t* bytes, const int32_t* offsets, int32_t n) {
    if (int rc = check_batch(c, bytes, offsets, n)) return rc;
    FG_CUDA(c, cudaSetDevice(c->device));
    if (n > 0) {
        const size_t b0 = (size_t)offsets[0], b1 = (size_t)offsets[n];
        FG_CUDA(c, cudaMemcpy(c->d_bytes + b0, bytes + b0, b1 - b0, cudaMemcpyHostToDevice));
        FG_CUDA(c, cudaMemcpy(c->offsets.d, offsets, sizeof(int32_t) * ((size_t)n + 1), cudaMemcpyHostToDevice));
        c->res_bytes = b1 - b0;
    } else {
        c->res_bytes = 0;
    }
    FG_CUDA(c, cudaMemset(c->d_k, 0, sizeof(uint32_t) * fg::K5_COUNT));
    FG_CUDA(c, fg::launch_check_offsets(c->offsets.dev<int32_t>(), n, (long long)c->max_bytes, c->d_k + fg::K5_BAD_OFFSETS, c->s_comp));
    uint32_t bad = 0;
    FG_CUDA(c, cudaMemcpyAsync(&bad, c->d_k + fg::K5_BAD_OFFSETS, 4, cudaMemcpyDeviceToHost, c->s_comp));
    FG_CUDA(c, cudaStreamSynchronize(c->s_comp));
    if (bad) return fail(c, FG_E_ARG, kBadOffsets);
    c->res_n = n;
    c->res_fmt = -1;
    return FG_OK;
}

int fg_parse_resident(fg_ctx* c, fg_format fmt, float* kernel_ms) {
    if (!c) return FG_E_ARG;
    if ((int)fmt < 0 || (int)fmt > 3) return fail(c, FG_E_ARG, "unknown format");
    FG_CUDA(c, cudaSetDevice(c->device));
    if (int rc = ensure_format(c, (int)fmt)) return rc;
    c->call_year = current_year(c);
    for (int attempt = 0; attempt < 2; ++attempt) {
        FG_CUDA(c, cudaMemsetAsync(c->d_k, 0, sizeof(uint32_t) * fg::K5_BAD_OFFSETS, c->s_comp));
        FG_CUDA(c, cudaEventRecord(c->ev_a, c->s_comp));
        if (int rc = launch_lines(c, (int)fmt, 0, c->res_n, pick_tile(c, c->res_bytes, c->res_n, (int)fmt), nullptr, 0, c->s_comp, true)) return rc;
        FG_CUDA(c, cudaEventRecord(c->ev_b, c->s_comp));
        uint32_t total[fg::K5_COUNT] = {};
        FG_CUDA(c, cudaMemcpyAsync(total, c->d_k, sizeof total, cudaMemcpyDeviceToHost, c->s_comp));
        FG_CUDA(c, cudaStreamSynchronize(c->s_comp));
        if (tables_overflow(c, (int)fmt, total)) {
            if (int rc = regrow_tables(c, (int)fmt, total)) return rc;
            continue;
        }
        float ms = 0.f;
        FG_CUDA(c, cudaEventElapsedTime(&ms, c->ev_a, c->ev_b));
        if (kernel_ms) *kernel_ms = ms;
        FG_CUDA(c, cudaEventElapsedTime(&c->last_dom_ms, c->ev_dom0, c->ev_dom1));
        c->res_fmt = (int)fmt;
        memcpy(c->res_tot, total, sizeof total);
        return FG_OK;
    }
    return fail(c, FG_E_CAPACITY, "side table overflow after regrow");
}

// K back-to-back passes over the resident batch with ONE host synchronisation at the end (what bench.py times):
// total_ms = CUDA-event time from before the first launch to after the last one.
int fg_parse_resident_n(fg_ctx* c, fg_format fmt, int32_t k, float* total_ms) {
    if (!c || k < 1) return FG_E_ARG;
    if ((int)fmt < 0 || (int)fmt > 3) return fail(c, FG_E_ARG, "unknown format");
    FG_CUDA(c, cudaSetDevice(c->device));
    if (int rc = ensure_format(c, (int)fmt)) return rc;
    c->call_year = current_year(c);
    // the side tables must already be large enough (one fg_parse_resident warm-up regrows them): checked after the loop
    const int tile = pick_tile(c, c->res_bytes, c->res_n, (int)fmt);
    FG_CUDA(c, cudaEventRecord(c->ev_a, c->s_comp));
    for (int32_t it = 0; it < k; ++it) {
        FG_CUDA(c, cudaMemsetAsync(c->d_k, 0, sizeof(uint32_t) * fg::K5_BAD_OFFSETS, c->s_comp));
        if (int rc = launch_lines(c, (int)fmt, 0, c->res_n, tile, nullptr, 0, c->s_comp)) return rc;
    }
    FG_CUDA(c, cudaEventRecord(c->ev_b, c->s_comp));
    uint32_t total[fg::K5_COUNT] = {};
    FG_CUDA(c, cudaMemcpyAsync(total, c->d_k, sizeof total, cudaMemcpyDeviceToHost, c->s_comp));
    FG_CUDA(c, cudaStreamSynchronize(c->s_comp));
    if (tables_overflow(c, (int)fmt, total))
        return fail(c, FG_E_CAPACITY, "side table too small: call fg_parse_resident once before fg_parse_resident_n");
    float ms = 0.f;
    FG_CUDA(c, cudaEventElapsedTime(&ms, c->ev_a, c->ev_b));
    if (total_ms) *total_ms = ms;
    c->res_fmt = (int)fmt;
    memcpy(c->res_tot, total, sizeof total);
    return FG_OK;
}

int fg_download(fg_ctx* c, fg_format fmt, fg_batch_out* out) {
    if (!c || !out) return FG_E_ARG;
    if (c->res_fmt != (int)fmt) return fail(c, FG_E_ARG, "no resident parse of this format to download");
    FG_CUDA(c, cudaSetDevice(c->device));
    memset(out, 0, sizeof *out);
    const uint32_t zero[fg::K5_COUNT] = {};
    if (int rc = copy_rows_d2h(c, fmt, 0, c->res_n, c->s_d2h)) return rc;
    if (int rc = copy_tables_d2h(c, fmt, zero, c->res_tot)) return rc;
    FG_CUDA(c, cudaStreamSynchronize(c->s_d2h));
    fill_out(c, fmt, c->res_n, c->res_tot, out);
    return FG_OK;
}

int fg_flush_l2(fg_ctx* c) {
    if (!c) return FG_E_ARG;
    FG_CUDA(c, cudaSetDevice(c->device));
    if (!c->d_flush) FG_CUDA(c, cudaMalloc(&c->d_flush, kL2FlushBytes));
    FG_CUDA(c, cudaMemsetAsync(c->d_flush, 0x5A, kL2FlushBytes, c->s_comp));
    FG_CUDA(c, cudaStreamSynchronize(c->s_comp));
    return FG_OK;
}

const char* fg_error_string(fg_format, uint32_t status) {
    if (status == 0 || status >= FG_ST_COUNT) return nullptr;
    return kErrorStrings[status];
}
uint32_t fg_error_count(void) { return FG_ST_COUNT; }

const char* fg_build_info(void) { return fg::kernel_build_info(); }
int64_t fg_kernel_launches(const fg_ctx* c) { return c ? c->launches : 0; }
float fg_last_split_ms(const fg_ctx* c) { return c ? c->last_split_ms : 0.f; }
float fg_last_dominant_kernel_ms(const fg_ctx* c) { return c ? c->last_dom_ms : 0.f; }

}  // extern "C"
