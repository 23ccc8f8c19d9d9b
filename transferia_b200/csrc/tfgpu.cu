// C-ABI of the B200 columnar transform engine (include/tfgpu.h). Host orchestration only: every
// per-row operation runs in the sm_100a kernels of kernels_*.cuh.  There is no CPU fallback: without
// a CUDA device tfgpu_engine_create fails with TF_E_FATAL_NODEVICE.
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/tfgpu.h"
#include "../../include/tfgpu_sink.h"
#include "plan.hpp"
#include "device_types.cuh"
#include "launch.hpp"

using namespace tfk;

namespace {

struct CudaError { cudaError_t e; const char* what; };
#define CK(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) throw CudaError{_e, #x}; } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct DevBuf {
    uint8_t* p = nullptr; size_t cap = 0;
    void ensure(size_t n) {
        if (n <= cap) return;
        if (p) { CK(cudaDeviceSynchronize()); CK(cudaFree(p)); p = nullptr; cap = 0; }
        size_t want = align_up(n + n / 8 + 4096, 1 << 20);
        CK(cudaMalloc(&p, want)); cap = want;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PlanDev {
    tfplan::Plan plan;
    // device copies of plan constants
    DevBuf consts;
    DTerm* d_terms = nullptr; uint32_t* d_expr_off = nullptr; DFilterStep* d_fsteps = nullptr; uint8_t* d_blob = nullptr;
    uint8_t* d_col_headers = nullptr; uint32_t* d_col_header_off = nullptr;
    JsonCol* d_jcols = nullptr; uint8_t* d_jnames = nullptr; size_t jnames_len = 0;
    JsonCol* d_sjcols = nullptr; JsonCol* d_scsvcols = nullptr; uint8_t* d_snames = nullptr;      // batch serializers: sorted JSON keys (pre-quoted), CSV order
    int32_t* d_fixed_slots = nullptr; int32_t* d_str_slots = nullptr; int32_t* d_mask_slots = nullptr; int32_t* d_out_cols = nullptr;
    MaskKey* d_mask_keys = nullptr;
    int n_fsteps = 0, n_fixed_slots = 0, n_str = 0, n_mask_cols = 0, n_tostr = 0;
    std::vector<int32_t> fixed_slots, str_slots, mask_slot_cols, mask_slot_key;
    std::vector<int> col_out_kind, col_out_w, col_str_slot, col_mask_slot, col_nullable;
    ShardCol* d_shard_cols = nullptr;              // sharder_transformer: columns it reads (plan.has_sharder)
    std::vector<JsonCol> h_sjcols;                 // host copy of d_sjcols (the Debezium emitter picks the key columns out of it)
    DevBuf dbz_consts; std::string dbz_opts_key; DbzEmitArgs dbz{};      // Debezium emitter: message template of the last opts_json
};

}  // namespace

struct tfgpu_engine {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr, side_stream = nullptr;   // side_stream: string encode runs beside the fixed-width encode
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // The checksum chain and the wire gather of an LZ4 batch run on two side streams and are NOT joined at the end of the call: the
    // next batch's filter / encode kernels overlap them (they only wait before they reuse the frame slots). join_tail() orders the
    // main stream after them; every path that reads results, changes layout or leaves the LZ4 format calls it.
    cudaStream_t side2_stream = nullptr; cudaEvent_t ev_tail2 = nullptr; bool tail_pending = false; uint64_t tail_nrows = 0, tail_nframes_max = 0; const void* tail_plan = nullptr;
    uint64_t* d_tail = nullptr;
    std::string last_error;
    uint64_t launches = 0;
    uint32_t frame_bytes = LZ_MAX_FRAME;
    int sm_count = 148;
    std::vector<std::unique_ptr<PlanDev>> plans;
    // arenas
    DevBuf in_arena, work, raw, slots, wire, strict_stage, lens_arena, lens_arena2, csv_text, csv_stage, json_msgs, n2f_stage, n2f_heap, off_scratch;
    DState* d_state = nullptr; DCol* d_cols = nullptr; size_t d_cols_cap = 0;
    int32_t* d_call_slots = nullptr; ColRegions* d_regions = nullptr; size_t d_call_cap = 0;   // columnar mode, per call
    // pointers into `work` for the last call
    uint8_t *keep = nullptr, *errcode = nullptr, *errstep = nullptr; uint32_t *blockcnt = nullptr, *blockoff = nullptr, *sel = nullptr;
    uint32_t* tile_sum = nullptr; uint64_t* tile_base = nullptr; uint64_t* col_bytes = nullptr; uint32_t* comp_size = nullptr; uint64_t* wire_off = nullptr; unsigned long long* frame_pfx = nullptr;
    uint64_t last_nrows = 0; bool last_has_filter = false, last_has_sharder = false; int last_wire_fmt = 0;
    uint8_t* pinned = nullptr; size_t pinned_cap = 0;
    // two-phase push (tfgpu_push_encode_selective): device flags of phase one, their pinned host copy, the host gather's buffers
    DevBuf err_list;                                   // fetch_errors: counter + (row, code, term) triples
    DevBuf sel_stage; uint8_t* sel_host = nullptr; size_t sel_host_cap = 0; tfgpu_columnar* gather_pool = nullptr;
    uint64_t h2d_bytes = 0;                            // bytes stage_input has copied to the device since creation
    DevBuf json_sizes, dbz_keysz, dbz_meta, dbz_old, dbz_msgsz, old_arena, part_ids;
    DbzEmitArgs dbz{};                                 // set by tfgpu_emit_debezium for the TF_WIRE_DEBEZIUM branch of run_chain
    unsigned long long* lz_phases = nullptr;      // debug: per-phase cycle counters of k_lz4_frames
    void* work_json_sizes(uint64_t n) { json_sizes.ensure(n * 4 + 256); return json_sizes.p; }
    // optional per-kernel CUDA-event timing of the last call (bench roofline)
    bool prof_on = false; std::vector<cudaEvent_t> prof_ev; std::vector<const char*> prof_names; int prof_n = 0;
    std::string prof_json;
    void prof_begin(const char* name, cudaStream_t s) {
        launches++;
        if (!prof_on) return;
        while ((int)prof_ev.size() < 2 * (prof_n + 1)) { cudaEvent_t ev; cudaEventCreate(&ev); prof_ev.push_back(ev); }
        if ((int)prof_names.size() <= prof_n) prof_names.resize(prof_n + 1);
        prof_names[prof_n] = name; cudaEventRecord(prof_ev[2 * prof_n], s);
    }
    void prof_end(cudaStream_t s) { if (!prof_on) return; cudaEventRecord(prof_ev[2 * prof_n + 1], s); prof_n++; }
};

struct tfgpu_result {
    uint64_t rows_in = 0, rows_out = 0, raw_len = 0, n_frames = 0, consumed = 0;
    std::vector<tf_rowerr> errs;
    uint8_t* bytes = nullptr; uint64_t bytes_len = 0; bool bytes_pinned = false;
    std::vector<uint32_t> selection;       // parsers: input row (line / message) of every output row
    std::vector<uint8_t> meta_kinds; std::vector<uint32_t> meta_tx; std::vector<uint64_t> meta_lsn, meta_ct;   // debezium: per message
    std::vector<uint32_t> row_sizes;       // row-text formats: bytes of every output row (incl. its separator / newline)
    std::vector<uint32_t> key_sizes;       // Debezium emitter: key message bytes of every output row
    std::vector<uint32_t> msg_sizes;       // Debezium emitter: 7 per output row — message count, then (key bytes, value bytes | 0xFFFFFFFF) per message
    std::vector<uint32_t> part_ids;        // sharder_transformer: ChangeItem.PartID (as an integer) of every output row
    // push_columns output
    tf_batch batch{}; std::vector<tf_col> cols; std::vector<uint8_t*> owned;
};

namespace {

void join_tail(tfgpu_engine* e) {
    if (!e->tail_pending) return;
    CK(cudaStreamWaitEvent(e->stream, e->ev_tail2, 0));
    e->tail_pending = false;
}
int fail(tfgpu_engine* e, int code, const std::string& msg) { if (e) e->last_error = msg; return code; }
int cuda_fail(tfgpu_engine* e, const CudaError& c) {
    std::string m = std::string("CUDA error: ") + cudaGetErrorString(c.e) + " in " + c.what;
    cudaGetLastError();
    return fail(e, c.e == cudaErrorMemoryAllocation ? TF_E_RETRY_OOM : TF_E_RETRY_LAUNCH, m);
}

// Body of an engine entry point: runs on the engine's device; what it throws becomes the call's return code and last_error
// (FatalError derives from std::runtime_error, so it is caught first).
template <class F> int guarded(tfgpu_engine* e, F&& body) {
    try {
        CK(cudaSetDevice(e->device));
        return body();
    } catch (const tfplan::FatalError& f) { return fail(e, f.code, f.what()); }
    catch (const CudaError& c) { return cuda_fail(e, c); }
    catch (const std::bad_alloc&) { return fail(e, TF_E_RETRY_OOM, "host allocation failed"); }
    catch (const std::exception& x) { return fail(e, TF_E_FATAL_CONFIG, x.what()); }
}

// Body of a host-only validator: `describe` builds the description, copied NUL-terminated into describe_out; what it throws
// becomes the return code (a FatalError's own, else TF_E_FATAL_CONFIG) with its text in err_out.
template <class F> int validated(char* describe_out, uint64_t cap, char* err_out, uint64_t err_cap, F&& describe) {
    auto put = [](char* dst, uint64_t cap_, const std::string& s) { if (dst && cap_) { size_t n = s.size() < cap_ - 1 ? s.size() : cap_ - 1; std::memcpy(dst, s.data(), n); dst[n] = 0; } };
    try {
        const std::string d = describe();
        if (describe_out && d.size() + 1 > cap) { put(err_out, err_cap, "describe buffer too small"); return TF_E_FATAL_ARG; }
        put(describe_out, cap, d);
        return TF_OK;
    } catch (const tfplan::FatalError& f) { put(err_out, err_cap, f.what()); return f.code; }
    catch (const std::exception& x) { put(err_out, err_cap, x.what()); return TF_E_FATAL_CONFIG; }
}

// encoding/json appendString with escapeHTML off, for column names (json.go:56-58)
std::string host_json_quote_nohtml(const std::string& in) {
    static const char* hex = "0123456789abcdef";
    std::string d = "\""; const uint8_t* s = (const uint8_t*)in.data(); const size_t n = in.size();
    for (size_t i = 0; i < n;) {
        const uint8_t b = s[i];
        if (b < 0x80) {
            if (b >= 0x20 && b != '"' && b != '\\') d += (char)b;
            else { d += '\\'; switch (b) { case '"': case '\\': d += (char)b; break; case '\b': d += 'b'; break; case '\f': d += 'f'; break; case '\n': d += 'n'; break; case '\r': d += 'r'; break; case '\t': d += 't'; break;
                                            default: d += "u00"; d += hex[b >> 4]; d += hex[b & 15]; } }
            i++; continue;
        }
        uint32_t r = 0xFFFD; size_t w = 1;
        if (b >= 0xC2 && b <= 0xDF && i + 1 < n && (s[i + 1] & 0xC0) == 0x80) { r = ((b & 0x1Fu) << 6) | (s[i + 1] & 0x3Fu); w = 2; }
        else if (b >= 0xE0 && b <= 0xEF && i + 2 < n && (s[i + 1] & 0xC0) == 0x80 && (s[i + 2] & 0xC0) == 0x80) { const uint32_t t = ((b & 0x0Fu) << 12) | ((s[i + 1] & 0x3Fu) << 6) | (s[i + 2] & 0x3Fu); if (t >= 0x800 && !(t >= 0xD800 && t <= 0xDFFF)) { r = t; w = 3; } }
        else if (b >= 0xF0 && b <= 0xF4 && i + 3 < n && (s[i + 1] & 0xC0) == 0x80 && (s[i + 2] & 0xC0) == 0x80 && (s[i + 3] & 0xC0) == 0x80) { const uint32_t t = ((b & 0x07u) << 18) | ((s[i + 1] & 0x3Fu) << 12) | ((s[i + 2] & 0x3Fu) << 6) | (s[i + 3] & 0x3Fu); if (t >= 0x10000 && t <= 0x10FFFF) { r = t; w = 4; } }
        if (r == 0xFFFD && w == 1) d += "\\ufffd";
        else if (r == 0x2028 || r == 0x2029) { d += "\\u202"; d += hex[r & 0xF]; }
        else d.append((const char*)s + i, w);
        i += w;
    }
    return d + "\"";
}

int in_width(int tf) {
    switch (tf) {
    case TF_INT8: case TF_UINT8: case TF_BOOLEAN: return 1;
    case TF_INT16: case TF_UINT16: return 2;
    case TF_INT32: case TF_UINT32: case TF_FLOAT: return 4;
    case TF_INT64: case TF_UINT64: case TF_DOUBLE: case TF_INTERVAL: case TF_DATE: case TF_DATETIME: case TF_TIMESTAMP: return 8;
    }
    return 0;
}

// Kernel descriptor of column `c` read as `type`, without an output kind or a String / mask slot
DCol plain_dcol(const tf_col& c, int type) {
    DCol d; std::memset(&d, 0, sizeof d);
    d.type = type; d.in_w = in_width(type); d.str_slot = -1; d.mask_slot = -1;
    d.values = (const uint8_t*)c.values; d.validity = c.validity; d.offsets = c.offsets; d.heap = c.heap; d.aux = (const uint8_t*)c.aux;
    return d;
}

template <typename T> T* carve(uint8_t*& p, size_t count) { T* r = (T*)p; p += align_up(count * sizeof(T), 256); return r; }

void upload_plan(tfgpu_engine* e, PlanDev& pd) {
    const tfplan::Plan& pl = pd.plan;
    const size_t nc = pl.in_schema.size();
    // which mask step (if any) owns each column
    pd.col_mask_slot.assign(nc, -1);
    std::vector<MaskKey> keys;
    for (size_t m = 0; m < pl.masks.size(); m++) {
        keys.push_back(make_mask_key((const uint8_t*)pl.masks[m].salt.data(), pl.masks[m].salt.size()));
        for (int c : pl.masks[m].cols) {
            if (pd.col_mask_slot[c] >= 0) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "column masked twice in one chain");
            pd.col_mask_slot[c] = (int)m;
        }
    }
    pd.col_out_kind.assign(nc, 0); pd.col_out_w.assign(nc, 0); pd.col_str_slot.assign(nc, -1);
    pd.col_nullable.assign(nc, 0);
    for (size_t k = 0; k < pl.out_cols.size(); k++) {
        const size_t c = (size_t)pl.out_cols[k];
        const int tf = pl.in_schema[c].tf;
        int kind, w;
        if (pd.col_mask_slot[c] >= 0) {
            kind = OK_MASK; w = 65;
        } else if (pl.tostr_col.size() > c && pl.tostr_col[c]) { kind = OK_TOSTR; w = 0; }
        else if (pl.todt_col.size() > c && pl.todt_col[c]) { kind = OK_TODT; w = 4; }
        else switch (tf) {
            case TF_BOOLEAN: kind = OK_BOOL; w = 1; break;
            case TF_DATE: kind = OK_DATE; w = 2; break;
            case TF_DATETIME: kind = OK_DATETIME; w = 4; break;
            case TF_TIMESTAMP: kind = OK_TS64; w = 8; break;
            case TF_BYTES: case TF_UTF8: case TF_ANY: kind = OK_STR; w = 0; break;
            default: kind = OK_COPY; w = in_width(tf);
        }
        pd.col_out_kind[c] = kind; pd.col_out_w[c] = w;
        const bool nullable = !pl.out_schema[k].required; pd.col_nullable[c] = nullable ? 1 : 0;
        if (kind == OK_STR || kind == OK_TOSTR) { pd.col_str_slot[c] = (int)pd.str_slots.size(); pd.str_slots.push_back((int32_t)c); }
        else if (kind == OK_MASK) { pd.mask_slot_cols.push_back((int32_t)c); }
        else pd.fixed_slots.push_back((int32_t)c);
        if (nullable && kind == OK_TODT) pd.fixed_slots.push_back((int32_t)c | TF_SLOT_ZEROMAP);
        else if (nullable && kind != OK_MASK && kind != OK_TOSTR) pd.fixed_slots.push_back((int32_t)c | TF_SLOT_NULLMAP);
    }
    if (pd.str_slots.size() > 256) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "more than 256 String columns");
    // JSONEachRow descriptors: column name + the ClickHouse class of the RESULT type (columntypes.ToChType)
    std::vector<JsonCol> jcols; std::vector<uint8_t> jnames;
    for (size_t k = 0; k < pl.out_cols.size(); k++) {
        JsonCol jc; std::memset(&jc, 0, sizeof jc); jc.col = pl.out_cols[k]; jc.name_off = (int32_t)jnames.size(); jc.name_len = (int32_t)pl.out_schema[k].name.size();
        jnames.insert(jnames.end(), pl.out_schema[k].name.begin(), pl.out_schema[k].name.end());
        const int rt = pl.out_schema[k].tf; jc.result_tf = rt;
        jc.ch_class = (rt == TF_ANY || rt == TF_BYTES || rt == TF_UTF8) ? JC_STRING : rt == TF_DATE ? JC_DATE : rt == TF_DATETIME ? JC_DATETIME : rt == TF_TIMESTAMP ? JC_DT64 : JC_OTHER;
        jc.prec = 6;
        jcols.push_back(jc);
    }
    pd.jnames_len = jnames.size();
    // batch serializers (pkg/serializer): encoding/json writes map keys sorted; the key text `"name":` is quoted here once
    std::vector<JsonCol> sjcols, scsvcols; std::vector<uint8_t> snames;
    {
        std::vector<size_t> order(pl.out_cols.size()); for (size_t k = 0; k < order.size(); k++) order[k] = k;
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return pl.out_schema[a].name < pl.out_schema[b].name; });
        for (size_t j = 0; j < order.size(); j++) {
            const size_t k = order[j]; JsonCol jc = jcols[k]; jc.pad0 = (int32_t)k;
            const std::string q = host_json_quote_nohtml(pl.out_schema[k].name) + ":";
            jc.name_off = (int32_t)snames.size(); jc.name_len = (int32_t)q.size(); snames.insert(snames.end(), q.begin(), q.end());
            sjcols.push_back(jc);
        }
        for (size_t k = 0; k < jcols.size(); k++) { JsonCol jc = jcols[k]; jc.pad0 = (int32_t)k; scsvcols.push_back(jc); }
        pd.h_sjcols = sjcols;
    }
    // flatten filter steps
    std::vector<DTerm> terms; std::vector<uint32_t> expr_off(1, 0); std::vector<DFilterStep> fsteps;
    for (size_t f = 0; f < pl.filters.size(); f++) {
        DFilterStep st; st.expr_begin = (int32_t)expr_off.size() - 1; st.nexpr = (int32_t)pl.filters[f].exprs.size(); st.step_index = pl.filter_step_index[f];
        st.flags = (pl.filters[f].is_skip ? 1 : 0) | (pl.filters[f].pass_all ? 2 : 0);
        if (pl.filters[f].is_skip) { st.expr_begin = pl.filters[f].kind_mask; st.nexpr = 0; }
        for (auto& ex : pl.filters[f].exprs) {
            for (auto& t : ex) { DTerm d; static_assert(sizeof(DTerm) == sizeof(tfplan::DTerm), "DTerm mismatch"); std::memcpy(&d, &t, sizeof d); terms.push_back(d); }
            expr_off.push_back((uint32_t)terms.size());
        }
        fsteps.push_back(st);
    }
    pd.n_fsteps = (int)fsteps.size(); pd.n_fixed_slots = (int)pd.fixed_slots.size(); pd.n_str = (int)pd.str_slots.size(); pd.n_mask_cols = (int)pd.mask_slot_cols.size();
    pd.n_tostr = 0; for (size_t c = 0; c < pd.col_out_kind.size(); c++) if (pd.col_out_kind[c] == OK_TOSTR) pd.n_tostr++;
    size_t total = 0;
    auto need = [&](size_t n) { total += align_up(n ? n : 1, 256); };
    need(terms.size() * sizeof(DTerm)); need(expr_off.size() * 4); need(fsteps.size() * sizeof(DFilterStep)); need(pl.blob.size());
    need(pl.col_headers.size()); need(pl.col_header_off.size() * 4); need(pd.fixed_slots.size() * 4); need(pd.str_slots.size() * 4);
    need(pd.mask_slot_cols.size() * 4); need(keys.size() * sizeof(MaskKey)); need(pl.out_cols.size() * 4); need(jcols.size() * sizeof(JsonCol)); need(jnames.size());
    need(sjcols.size() * sizeof(JsonCol)); need(scsvcols.size() * sizeof(JsonCol)); need(snames.size());
    std::vector<ShardCol> shcols;
    for (size_t k = 0; k < pl.shard_cols.size(); k++) shcols.push_back(ShardCol{pl.shard_cols[k], pl.shard_form[k], 0, 0});
    need(shcols.size() * sizeof(ShardCol));
    pd.consts.ensure(total);
    uint8_t* p = pd.consts.p;
    auto put = [&](const void* src, size_t n) { uint8_t* d = p; if (n) CK(cudaMemcpy(d, src, n, cudaMemcpyHostToDevice)); p += align_up(n ? n : 1, 256); return d; };
    pd.d_terms = (DTerm*)put(terms.data(), terms.size() * sizeof(DTerm));
    pd.d_expr_off = (uint32_t*)put(expr_off.data(), expr_off.size() * 4);
    pd.d_fsteps = (DFilterStep*)put(fsteps.data(), fsteps.size() * sizeof(DFilterStep));
    pd.d_blob = put(pl.blob.data(), pl.blob.size());
    pd.d_col_headers = put(pl.col_headers.data(), pl.col_headers.size());
    pd.d_col_header_off = (uint32_t*)put(pl.col_header_off.data(), pl.col_header_off.size() * 4);
    pd.d_fixed_slots = (int32_t*)put(pd.fixed_slots.data(), pd.fixed_slots.size() * 4);
    pd.d_str_slots = (int32_t*)put(pd.str_slots.data(), pd.str_slots.size() * 4);
    pd.d_mask_slots = (int32_t*)put(pd.mask_slot_cols.data(), pd.mask_slot_cols.size() * 4);
    pd.d_mask_keys = (MaskKey*)put(keys.data(), keys.size() * sizeof(MaskKey));
    { std::vector<int32_t> oc(pl.out_cols.begin(), pl.out_cols.end()); pd.d_out_cols = (int32_t*)put(oc.data(), oc.size() * 4); }
    pd.d_jcols = (JsonCol*)put(jcols.data(), jcols.size() * sizeof(JsonCol)); pd.d_jnames = put(jnames.data(), jnames.size());
    pd.d_sjcols = (JsonCol*)put(sjcols.data(), sjcols.size() * sizeof(JsonCol)); pd.d_scsvcols = (JsonCol*)put(scsvcols.data(), scsvcols.size() * sizeof(JsonCol)); pd.d_snames = put(snames.data(), snames.size());
    pd.d_shard_cols = (ShardCol*)put(shcols.data(), shcols.size() * sizeof(ShardCol));
    (void)e;
}

struct Sizes { uint64_t raw_bound, n_frames_max, wire_bound; uint32_t ntiles_cap, nblocks; };

Sizes compute_sizes(const tfgpu_engine* e, const PlanDev& pd, const tf_batch* in, bool columnar = false, bool json = false) {
    const tfplan::Plan& pl = pd.plan; const uint64_t n = in->nrows;
    uint64_t raw = 64 + pl.col_headers.size();
    for (int oc : pl.out_cols) {
        const size_t c = (size_t)oc;
        if (pd.col_nullable[c]) raw += n;
        bool n2f = false; for (int q : pl.n2f_cols) if ((size_t)q == c) n2f = true;       // number_to_float may lengthen literals (1e20 -> 100000000000000000000)
        if (pd.col_out_kind[c] == OK_STR) raw += (n2f ? 6 : 1) * in->cols[c].heap_len + 5 * n;
        else if (pd.col_out_kind[c] == OK_TOSTR) raw += (in_width(in->cols[c].type) ? 40 * n : (n2f ? 36 : 6) * in->cols[c].heap_len + 8 * n) + 5 * n;   // longest text form (RFC3339Nano / %v float / \\u00XX-escaped JSON string)
        else raw += (uint64_t)pd.col_out_w[c] * n;
        if (columnar) raw += 8 * n + 4 * (n + 1) + n / 8 + 6 * 16 + (pd.col_out_kind[c] == OK_MASK ? 64 * n : 0);   // widest value, aux, offsets, bitmap, padding
        if (json) raw += (uint64_t)(pl.in_schema[c].name.size() + 4 + 48) * n + (in_width(in->cols[c].type) ? 0 : (n2f ? 36 : 6) * in->cols[c].heap_len);   // name, quotes, longest scalar text, escaped payload
    }
    Sizes s;
    s.raw_bound = raw + 256;
    s.n_frames_max = (raw + e->frame_bytes - 1) / e->frame_bytes + 1;
    s.wire_bound = s.n_frames_max * (uint64_t)(LZ_HDR + lz4_bound(e->frame_bytes)) + 1024;
    s.ntiles_cap = (uint32_t)((n + TF_STR_TILE - 1) / TF_STR_TILE + 1);
    s.nblocks = (uint32_t)((n + 255) / 256 + 1);
    return s;
}


// exclusive scan of the text-cell lengths of every var-width column: offsets[slot][row], col_total[slot]
static void launch_offsets(tfgpu_engine* e, const uint32_t* d_len, uint64_t nrows, uint32_t nslots, uint32_t* d_off, uint64_t* d_tot, cudaStream_t s) {
    const uint32_t nchunks = (uint32_t)((nrows + CSV_OFF_CHUNK - 1) / CSV_OFF_CHUNK);
    if (!nchunks || !nslots) { launch_k_csv_offsets(nslots ? nslots : 1, 1024, 0, s, d_len, nrows, d_off, d_tot); return; }
    e->off_scratch.ensure((size_t)nslots * nchunks * 8 + 256);
    uint64_t* cs = (uint64_t*)e->off_scratch.p;
    e->prof_begin("k_offsets_sum", s); launch_k_offsets_sum(dim3(nchunks, nslots), 1024, 0, s, d_len, nrows, nchunks, cs); e->prof_end(s);
    e->prof_begin("k_offsets_chunks", s); launch_k_offsets_chunks(nslots, 32, 0, s, cs, nchunks, d_tot); e->prof_end(s);
    e->prof_begin("k_offsets_write", s); launch_k_offsets_write(dim3(nchunks, nslots), 1024, 0, s, d_len, nrows, nchunks, cs, d_tot, d_off); e->prof_end(s);
}

// The device parsers (CSV, JSON lines, Debezium) type their input in two passes: pass one writes the fixed-width values and the
// byte length of every text cell, pass two copies the text cells into per-column heaps placed from those lengths. What lies between
// and after the passes is shared; the pass kernels and their arguments stay per parser.

// Layout of a staging arena: every region starts at a multiple of 256 bytes (an empty one still takes 256).
struct ArenaLayout {
    size_t total = 0;
    size_t operator()(size_t bytes) { const size_t at = total; total += align_up(bytes ? bytes : 1, 256); return at; }
};

// Text heaps of the var-width columns (slots) of a parsed batch
struct VarHeaps {
    std::vector<uint64_t> total, base; uint8_t* heap = nullptr;
    explicit VarHeaps(int nslots) : total(nslots ? nslots : 1, 0), base(nslots ? nslots : 1, 0) {}
};

// Between the passes: scans the cell lengths d_len [nslots][nrows] into offsets d_off [nslots][nrows + 1], reads the slot totals
// back (one synchronise), gives every slot a 16-byte-aligned base in in_arena and uploads the bases to d_base for pass two.
// in_arena is free during a parse: the parsed batch is device resident, so stage_input does not run.
void place_heaps(tfgpu_engine* e, VarHeaps& h, const uint32_t* d_len, uint64_t nrows, int nslots, uint32_t* d_off, uint64_t* d_tot, uint64_t* d_base, const char* what) {
    cudaStream_t s = e->stream;
    launch_offsets(e, d_len, nrows, (uint32_t)nslots, d_off, d_tot, s);
    CK(cudaMemcpyAsync(h.total.data(), d_tot, (size_t)nslots * 8, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
    uint64_t run = 0; for (int k = 0; k < nslots; k++) { h.base[k] = run; run += align_up(h.total[k], 16); }
    if (run >= (1ull << 32)) throw tfplan::FatalError(TF_E_FATAL_ARG, std::string(what) + ": a text column exceeds 4 GiB");
    e->in_arena.ensure(run + 256); h.heap = e->in_arena.p;
    CK(cudaMemcpyAsync(d_base, h.base.data(), (size_t)nslots * 8, cudaMemcpyHostToDevice, s));
}

// what pass one writes beside the values: validity bitmaps (JSON, Debezium), nanoseconds of time columns and tags of `any` columns (CSV, JSON)
void parsed_extras(const CsvColDev& h, tf_col& d) { d.aux = h.w ? (const void*)h.aux32 : h.aux8; }
void parsed_extras(const JsnColDev& h, tf_col& d) { d.aux = h.w ? (const void*)h.aux32 : h.aux8; d.validity = (const uint8_t*)h.validity; }
void parsed_extras(const DbzColDev& h, tf_col& d) { d.validity = (const uint8_t*)h.validity; }

// The parsed columns as the device-resident batch the chain reads (`dev` holds its columns); a text column takes its slot's
// offsets (d_off) and heap.
template <class ColDev> tf_batch parsed_batch(const std::vector<ColDev>& hc, uint64_t nrows, const uint32_t* d_off, const VarHeaps& h, std::vector<tf_col>& dev) {
    dev.assign(hc.size(), tf_col{});
    for (size_t c = 0; c < hc.size(); c++) {
        tf_col& d = dev[c]; d.type = hc[c].tf; parsed_extras(hc[c], d);
        if (hc[c].w) d.values = hc[c].values;
        else { const int k = hc[c].slot; d.offsets = d_off + (size_t)k * (nrows + 1); d.heap = h.heap ? h.heap + h.base[k] : nullptr; d.heap_len = h.total[k]; }
    }
    return tf_batch{nrows, (uint32_t)hc.size(), TF_MEM_DEVICE, dev.data(), nullptr};
}

// Launch the whole fused chain on e->stream. `cols_host` holds DEVICE pointers.
#define TF_WIRE_COLUMNAR_INTERNAL 100
// x-extent of a (tiles, slots) grid whose kernel strides over its tiles: enough CTAs for `waves` full waves of the device
// (resident CTAs per SM taken as 6 for the 256-thread encode kernels), never more than the tiles there can be
uint32_t grid_cap(const tfgpu_engine* e, uint32_t tiles_upper, uint32_t nslots, uint32_t waves) {
    const uint32_t want = ((uint32_t)e->sm_count * 6u * waves + nslots - 1) / (nslots ? nslots : 1);
    return std::max(1u, std::min(tiles_upper, std::max(want, 8u)));
}

void run_chain(tfgpu_engine* e, PlanDev& pd, const tf_batch* in, const tf_col* dev_cols, const uint8_t* dev_kinds, int wire_fmt, const uint8_t* pre_err = nullptr) {
    const bool columnar = wire_fmt == TF_WIRE_COLUMNAR_INTERNAL;
    const tfplan::Plan& pl = pd.plan;
    const size_t nc = pl.in_schema.size(); const uint64_t n = in->nrows;
    const int wire_base = wire_fmt == TF_WIRE_COLUMNAR_INTERNAL ? wire_fmt : (wire_fmt & 0xff);
    const bool dbz = wire_base == TF_WIRE_DEBEZIUM;
    const bool ser = wire_base == TF_WIRE_SER_JSON || wire_base == TF_WIRE_SER_CSV || dbz;
    const bool json_rows = wire_base == TF_WIRE_CH_JSONEACHROW || ser;
    if (ser) for (size_t c = 0; c < nc; c++) if (pd.col_out_kind[c] == OK_TOSTR && pl.in_schema[c].tf == TF_ANY)
        throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "serializer sinks after convert_to_string on an `any` column are not handled on the device");
    const Sizes sz = compute_sizes(e, pd, in, columnar, json_rows);
    cudaStream_t s = e->stream;
    // a pending checksum / gather tail may only stay in flight across a call that lays the work arena out identically
    if (e->tail_pending && !(wire_fmt == TF_WIRE_CH_NATIVE_LZ4 && n == e->tail_nrows && (const void*)&pd == e->tail_plan && sz.n_frames_max == e->tail_nframes_max)) join_tail(e);
    // work arena
    size_t wbytes = 0;
    auto need = [&](size_t b) { wbytes += align_up(b ? b : 1, 256); };
    need(n); need(n); need(n); need(sz.nblocks * 4); need(sz.nblocks * 4); need(n * 4);
    const size_t nslot_alloc = (size_t)(pd.n_str > 0 ? pd.n_str : 1);
    need(nslot_alloc * sz.ntiles_cap * 4); need(nslot_alloc * sz.ntiles_cap * 8);
    need(sz.n_frames_max * 4); need(sz.n_frames_max * 8); need(sz.n_frames_max * 8); need(256 * 8);
    e->work.ensure(wbytes);
    uint8_t* p = e->work.p;
    e->keep = carve<uint8_t>(p, n); e->errcode = carve<uint8_t>(p, n); e->errstep = carve<uint8_t>(p, n);
    e->blockcnt = carve<uint32_t>(p, sz.nblocks); e->blockoff = carve<uint32_t>(p, sz.nblocks); e->sel = carve<uint32_t>(p, n);
    e->tile_sum = carve<uint32_t>(p, nslot_alloc * sz.ntiles_cap); e->tile_base = carve<uint64_t>(p, nslot_alloc * sz.ntiles_cap);
    e->comp_size = carve<uint32_t>(p, sz.n_frames_max); e->wire_off = carve<uint64_t>(p, sz.n_frames_max); e->frame_pfx = carve<unsigned long long>(p, sz.n_frames_max); e->col_bytes = carve<uint64_t>(p, 256);
    e->raw.ensure(sz.raw_bound);
    const bool lz = wire_fmt == TF_WIRE_CH_NATIVE_LZ4;
    if (lz) e->wire.ensure(sz.wire_bound);
    if (e->d_cols_cap < nc) { if (e->d_cols) CK(cudaFree(e->d_cols)); CK(cudaMalloc(&e->d_cols, sizeof(DCol) * nc)); e->d_cols_cap = nc; }
    // column descriptors
    std::vector<DCol> hc(nc); std::vector<StrictCol> strict;
    for (size_t c = 0; c < nc; c++) {
        const tf_col& ic = dev_cols[c]; DCol& d = hc[c]; std::memset(&d, 0, sizeof d);
        int ctype = ic.type;
        if (ic.type != pl.in_schema[c].tf) {        // a loose value type: Strictify it to the column's type first (strictify.go:46-157)
            const int st = ic.type, dt = pl.in_schema[c].tf;
            const bool s_num = in_width(st) && st != TF_INTERVAL && st != TF_DATE && st != TF_DATETIME && st != TF_TIMESTAMP;
            if ((st == TF_UTF8 && dt == TF_BYTES) || (st == TF_BYTES && dt == TF_UTF8)) ctype = dt;      // castx.ToByteSliceE(string) / ToStringE([]byte): the same bytes
            else if (s_num && in_width(dt) && !(st == TF_FLOAT && dt == TF_DOUBLE) && !(st == TF_BOOLEAN && dt == TF_DOUBLE)) { strict.push_back(StrictCol{(const uint8_t*)ic.values, nullptr, ic.validity, st, dt, (int32_t)c, 0}); ctype = dt; }
            else throw tfplan::FatalError(TF_E_FATAL_ARG, "column " + std::to_string(c) + ": a " + std::to_string(st) + " value cannot be strictified to the plan's column type on the device");
        }
        d.type = ctype; d.out_kind = pd.col_out_kind[c]; d.in_w = in_width(ctype); d.out_w = pd.col_out_w[c];
        if (columnar && d.out_kind == OK_TODT) d.out_w = 8;          // Transformed value is a time.Time: int64 seconds
        else if (columnar && d.out_kind != OK_STR && d.out_kind != OK_MASK && d.out_kind != OK_TOSTR) { d.out_kind = OK_COPY; d.out_w = d.in_w; }   // Transformed values keep their type
        d.nullable = pd.col_nullable[c]; d.str_slot = pd.col_str_slot[c]; d.mask_slot = pd.col_mask_slot[c];
        d.values = (const uint8_t*)ic.values; d.validity = ic.validity; d.offsets = ic.offsets; d.heap = ic.heap; d.aux = (const uint8_t*)ic.aux;
        if (n) {
            if (d.in_w && !d.values) throw tfplan::FatalError(TF_E_FATAL_ARG, "column " + std::to_string(c) + ": values pointer is NULL");
            if (!d.in_w && !d.offsets) throw tfplan::FatalError(TF_E_FATAL_ARG, "column " + std::to_string(c) + ": offsets pointer is NULL");
        }
    }
    if (!pre_err) e->prof_n = 0;
    const uint8_t* pre_term = nullptr;
    if (!strict.empty() && n) {        // Strictify pre-pass: loose fixed-width values -> the schema's type, range / cast failures as row errors
        size_t sb = 0; auto need3 = [&](size_t b) { size_t at = sb; sb += align_up(b ? b : 1, 256); return at; };
        const size_t o_desc = need3(strict.size() * sizeof(StrictCol)), o_err = need3(n), o_term = need3(n);
        std::vector<size_t> o_val(strict.size());
        for (size_t k = 0; k < strict.size(); k++) o_val[k] = need3((size_t)in_width(strict[k].dst_tf) * n + 16);
        e->strict_stage.ensure(sb + 256);
        uint8_t* B = e->strict_stage.p;
        for (size_t k = 0; k < strict.size(); k++) { strict[k].dst = B + o_val[k]; hc[strict[k].col].values = B + o_val[k]; }
        CK(cudaMemcpyAsync(B + o_desc, strict.data(), strict.size() * sizeof(StrictCol), cudaMemcpyHostToDevice, s));
        if (pre_err) CK(cudaMemcpyAsync(B + o_err, pre_err, n, cudaMemcpyDeviceToDevice, s)); else CK(cudaMemsetAsync(B + o_err, 0, n, s));
        CK(cudaMemsetAsync(B + o_term, 0xff, n, s));
        StrictArgs sa{(const StrictCol*)(B + o_desc), (int)strict.size(), n, B + o_err, B + o_term};
        e->prof_begin("k_strictify", s); launch_k_strictify((uint32_t)((n + 255) / 256), 256, 0, s, sa); e->prof_end(s);
        pre_err = B + o_err; pre_term = B + o_term;
    }
    CK(cudaMemcpyAsync(e->d_cols, hc.data(), sizeof(DCol) * nc, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(e->d_state, 0, sizeof(DState), s));
    if (!pl.n2f_cols.empty() && n) {        // number_to_float: rewrite the JSON text of the `any` columns before anything reads them
        const size_t k2 = pl.n2f_cols.size();
        size_t sb = 0; auto need2 = [&](size_t b) { size_t at = sb; sb += align_up(b ? b : 1, 256); return at; };
        const size_t o_which = need2(k2 * 4), o_len = need2(k2 * n * 4), o_off = need2(k2 * (n + 1) * 4), o_tot = need2(k2 * 8 + 8), o_base = need2(k2 * 8 + 8), o_err = need2(n);
        e->n2f_stage.ensure(sb + 256);
        uint8_t* B = e->n2f_stage.p;
        std::vector<int32_t> which(pl.n2f_cols.begin(), pl.n2f_cols.end());
        CK(cudaMemcpyAsync(B + o_which, which.data(), k2 * 4, cudaMemcpyHostToDevice, s));
        if (pre_err) CK(cudaMemcpyAsync(B + o_err, pre_err, n, cudaMemcpyDeviceToDevice, s)); else CK(cudaMemsetAsync(B + o_err, 0, n, s));
        N2fArgs na{e->d_cols, (const int32_t*)(B + o_which), dev_kinds, n, (uint32_t*)(B + o_len), (const uint32_t*)(B + o_off), nullptr, (const uint64_t*)(B + o_base), B + o_err};
        e->prof_begin("k_n2f_sizes", s); launch_k_n2f_sizes(dim3((uint32_t)((n + 127) / 128), (uint32_t)k2), 128, 0, s, na); e->prof_end(s);
        launch_offsets(e, (const uint32_t*)(B + o_len), n, (uint32_t)k2, (uint32_t*)(B + o_off), (uint64_t*)(B + o_tot), s);
        std::vector<uint64_t> tot(k2), base(k2);
        CK(cudaMemcpyAsync(tot.data(), B + o_tot, k2 * 8, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
        uint64_t run = 0; for (size_t k = 0; k < k2; k++) { base[k] = run; run += align_up(tot[k], 16); }
        if (run >= (1ull << 32)) throw tfplan::FatalError(TF_E_FATAL_ARG, "number_to_float: a rewritten column exceeds 4 GiB");
        e->n2f_heap.ensure(run + 256);
        CK(cudaMemcpyAsync(B + o_base, base.data(), k2 * 8, cudaMemcpyHostToDevice, s));
        na.heap = e->n2f_heap.p;
        e->prof_begin("k_n2f_write", s); launch_k_n2f_write(dim3((uint32_t)((n + 127) / 128), (uint32_t)k2), 128, 0, s, na); e->prof_end(s);
        for (size_t k = 0; k < k2; k++) { DCol& d = hc[pl.n2f_cols[k]]; d.offsets = (const uint32_t*)(B + o_off) + k * (n + 1); d.heap = e->n2f_heap.p + base[k]; }
        CK(cudaMemcpyAsync(e->d_cols, hc.data(), sizeof(DCol) * nc, cudaMemcpyHostToDevice, s));
        pre_err = B + o_err;                 // parser errors carried over + N2F_HOST rows
    }
    // sink / serializer wire formats take INSERT rows only on the device (sink_table.go:296-305 refuses the others on non-updatable
    // tables, marshal.go:92-95 and the queue serializers need OldKeys): update / delete rows that survive the chain come back as row errors
    const bool sink_guard = dev_kinds && wire_fmt != TF_WIRE_COLUMNAR_INTERNAL && wire_base != TF_WIRE_DEBEZIUM;
    const bool has_filter = pd.n_fsteps > 0 || pre_err || sink_guard;
    e->last_nrows = n; e->last_has_filter = has_filter; e->last_wire_fmt = wire_fmt;
    const uint32_t nb = (uint32_t)((n + 255) / 256);
    if (has_filter && n) {
        FilterArgs fa{e->d_cols, dev_kinds, n, pd.d_fsteps, pd.n_fsteps, pd.d_expr_off, pd.d_terms, pd.d_blob, e->keep, e->errcode, e->errstep, e->blockcnt, e->d_state, pre_err, pre_term, sink_guard ? 1 : 0};
        e->prof_begin("k_filter", s); launch_k_filter(nb, 256, 0, s, fa); e->prof_end(s);
        e->prof_begin("k_scan_blockcnt", s); launch_k_scan_blockcnt(1, 1024, 0, s, e->blockcnt, e->blockoff, nb, e->d_state); e->prof_end(s);
        e->prof_begin("k_compact_sel", s); launch_k_compact_sel(nb, 256, 0, s, e->keep, e->blockoff, n, e->sel); e->prof_end(s);
    }
    const uint32_t* sel = (has_filter && n) ? e->sel : nullptr;
    const uint32_t ntiles = (uint32_t)((n + TF_STR_TILE - 1) / TF_STR_TILE);
    // (the string kernels keep one CTA per tile group and exit early past the kept rows: a capped grid with a stride loop
    // makes the CTAs of the heavy columns run several groups back to back; measured 0.18 -> 0.25 ms on the headline batch)
    const uint32_t str_gx = std::max(1u, (ntiles + TF_STR_GROUP - 1) / TF_STR_GROUP);
    EncodeArgs ea{e->d_cols, pd.d_str_slots, sel, e->d_state, e->raw.p, e->tile_sum, e->tile_base, sz.ntiles_cap, columnar ? 1 : 0};
    if (!has_filter || !n) {
        // n_kept = nrows is set inside k_layout (has_sel = 0); k_str_sizes needs it earlier:
        DState init; std::memset(&init, 0, sizeof init); init.n_kept = n;
        CK(cudaMemcpyAsync(e->d_state, &init, sizeof init, cudaMemcpyHostToDevice, s));
    }
    if (pl.has_sharder && n) {
        e->part_ids.ensure(n * 4 + 256);
        ShardArgs sa{e->d_cols, pd.d_shard_cols, (int)pl.shard_cols.size(), pd.d_mask_keys, sel, e->d_state, pl.shards, (uint32_t*)e->part_ids.p};
        e->prof_begin("k_shard_ids", s); launch_k_shard_ids(nb, 256, 0, s, sa); e->prof_end(s);
    }
    e->last_has_sharder = pl.has_sharder;
    if (json_rows) {
        // JSONEachRow: rows sized, placed by a tile scan, then written (kernels_json_out.cuh)
        const uint32_t jt = (uint32_t)((n + TF_JSON_TILE - 1) / TF_JSON_TILE);
        JsonArgs ja{e->d_cols, ser ? (wire_base == TF_WIRE_SER_CSV ? pd.d_scsvcols : pd.d_sjcols) : pd.d_jcols, (int)pl.out_cols.size(), ser ? pd.d_snames : pd.d_jnames, pd.d_mask_keys, sel, e->d_state, e->raw.p,
                    (uint32_t*)e->work_json_sizes(n), e->tile_sum, e->tile_base, e->col_bytes,
                    dbz ? 3 : ser ? (wire_base == TF_WIRE_SER_JSON ? 1 : 2) : 0, (uint32_t)(((wire_fmt & TF_WIRE_F_CLOSING_NEWLINE) ? TF_SER_NL : 0) | ((wire_fmt & TF_WIRE_F_ANY_AS_STRING) ? TF_SER_AAS : 0)), e->errcode, e->errstep, DbzEmitArgs{}};
        if (dbz) { ja.jcols = pd.d_sjcols; e->dbz_keysz.ensure(n * 4 + 256); e->dbz_msgsz.ensure(n * 28 + 256); ja.dz = e->dbz; ja.dz.key_size = (uint32_t*)e->dbz_keysz.p; ja.dz.msg_size = (uint32_t*)e->dbz_msgsz.p; }
        if (ser && !has_filter && n) { CK(cudaMemsetAsync(e->errcode, 0, n, s)); CK(cudaMemsetAsync(e->errstep, 0, n, s)); }
        if (jt) { e->prof_begin("k_json_sizes", s); launch_k_json_sizes(jt, TF_JSON_TILE, 0, s, ja); e->prof_end(s); }
        LayoutArgs lj{e->d_cols, 0, pd.d_out_cols, pd.d_str_slots, 1, e->tile_sum, e->tile_base, sz.ntiles_cap, pd.d_col_headers, pd.d_col_header_off,
                      e->raw.p, e->d_state, n, 1, e->frame_bytes, e->col_bytes};
        e->prof_begin("k_layout_scan", s); launch_k_layout_scan(1, 1024, 0, s, lj); e->prof_end(s);
        {   // row text has no useful upper bound ('f' floats reach 300+ characters): size the output from the measured total
            uint64_t total = 0; CK(cudaMemcpyAsync(&total, e->col_bytes, 8, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
            e->raw.ensure(total + 256); ja.raw = e->raw.p;
        }
        e->prof_begin("k_json_write", s); launch_k_json_write(jt ? jt : 1, TF_JSON_TILE, 0, s, ja); e->prof_end(s);
        CK(cudaGetLastError());
        return;
    }
    if (pd.n_str && ntiles) { e->prof_begin("k_str_sizes", s); launch_k_str_sizes(dim3(str_gx, pd.n_str), TF_STR_THREADS, 0, s, ea); e->prof_end(s); }
    LayoutArgs la{e->d_cols, (int)pl.out_cols.size(), pd.d_out_cols, pd.d_str_slots, pd.n_str, e->tile_sum, e->tile_base, sz.ntiles_cap, pd.d_col_headers, pd.d_col_header_off,
                  e->raw.p, e->d_state, n, 1, e->frame_bytes, e->col_bytes};
    if (pd.n_str) { e->prof_begin("k_layout_scan", s); launch_k_layout_scan(pd.n_str, 1024, 0, s, la); e->prof_end(s); }
    if (!columnar) {
        e->prof_begin("k_layout_finish", s); launch_k_layout_finish(1, 256, 0, s, la); e->prof_end(s);
        if (n) {
            // (the fixed-width streams and the String columns write disjoint parts of the block, but running them on two streams
            // was measured slower: both are latency-bound gathers that already fill the SMs: 0.087 + 0.182 ms in sequence, 0.30 ms side by side)
            if (pd.n_fixed_slots) {
                // widest stream is 8 bytes per row: words = 2n (+1 for misalignment)
                const uint32_t gx = grid_cap(e, (uint32_t)((2 * n + 2 + TF_FIX_TILE_WORDS - 1) / TF_FIX_TILE_WORDS), (uint32_t)pd.n_fixed_slots, 6);
                EncodeArgs fa = ea; fa.slots = pd.d_fixed_slots;
                e->prof_begin("k_encode_fixed", s); launch_k_encode_fixed(dim3(gx, pd.n_fixed_slots), 256, 0, s, fa); e->prof_end(s);
            }
            if (pd.n_str) { e->prof_begin("k_encode_str_plain", s); launch_k_encode_str_plain(dim3(str_gx, pd.n_str), TF_STR_THREADS, 0, s, ea); e->prof_end(s); }
            if (pd.n_str && pd.n_tostr) { e->prof_begin("k_encode_str", s); launch_k_encode_str(dim3(ntiles, pd.n_str), TF_STR_THREADS, 0, s, ea); e->prof_end(s); }
            if (pd.n_mask_cols) {
                MaskArgs ma{e->d_cols, pd.d_mask_slots, pd.d_mask_keys, sel, e->d_state, e->raw.p, 0};
                e->prof_begin("k_mask_encode", s); launch_k_mask_encode(dim3((uint32_t)((n + 127) / 128), pd.n_mask_cols), 128, 0, s, ma); e->prof_end(s);
            }
        }
    } else {
        // Transformed rows back in tf_batch layout (tfgpu_push_columns)
        const size_t no = pl.out_cols.size();
        if (e->d_call_cap < no) {
            if (e->d_call_slots) { CK(cudaFree(e->d_call_slots)); CK(cudaFree(e->d_regions)); }
            CK(cudaMalloc(&e->d_call_slots, sizeof(int32_t) * 3 * no)); CK(cudaMalloc(&e->d_regions, sizeof(ColRegions) * no)); e->d_call_cap = no;
        }
        std::vector<int32_t> fixed, valid;
        for (int oc : pl.out_cols) {
            const DCol& d = hc[oc];
            if (d.out_kind == OK_COPY || d.out_kind == OK_TODT) fixed.push_back(oc);
            const bool fresh = d.out_kind == OK_MASK || d.out_kind == OK_TOSTR || d.out_kind == OK_TODT;
            if (!fresh && d.aux) fixed.push_back(oc | TF_SLOT_AUX);
            if (!fresh && d.validity) valid.push_back(oc);
        }
        std::vector<int32_t> both(fixed); both.insert(both.end(), valid.begin(), valid.end());
        if (!both.empty()) CK(cudaMemcpyAsync(e->d_call_slots, both.data(), both.size() * 4, cudaMemcpyHostToDevice, s));
        e->prof_begin("k_layout_columnar", s); launch_k_layout_columnar(1, 256, 0, s, la, e->d_regions); e->prof_end(s);
        if (n) {
            if (!fixed.empty()) {
                const uint32_t gx = grid_cap(e, (uint32_t)((2 * n + 2 + TF_FIX_TILE_WORDS - 1) / TF_FIX_TILE_WORDS), (uint32_t)fixed.size(), 6);
                EncodeArgs fa = ea; fa.slots = e->d_call_slots;
                e->prof_begin("k_encode_fixed", s); launch_k_encode_fixed(dim3(gx, (uint32_t)fixed.size()), 256, 0, s, fa); e->prof_end(s);
            }
            if (!valid.empty()) {
                EncodeArgs va = ea; va.slots = e->d_call_slots + fixed.size();
                e->prof_begin("k_pack_validity", s); launch_k_pack_validity(dim3((uint32_t)((n / 8 + 256) / 256), (uint32_t)valid.size()), 256, 0, s, va); e->prof_end(s);
            }
            if (pd.n_str) { e->prof_begin("k_encode_str_plain", s); launch_k_encode_str_plain(dim3(str_gx, pd.n_str), TF_STR_THREADS, 0, s, ea); e->prof_end(s); }
            if (pd.n_str && pd.n_tostr) { e->prof_begin("k_encode_str", s); launch_k_encode_str(dim3(ntiles, pd.n_str), TF_STR_THREADS, 0, s, ea); e->prof_end(s); }
            if (pd.n_mask_cols) {
                MaskArgs ma{e->d_cols, pd.d_mask_slots, pd.d_mask_keys, sel, e->d_state, e->raw.p, 1};
                e->prof_begin("k_mask_encode", s); launch_k_mask_encode(dim3((uint32_t)((n + 127) / 128), pd.n_mask_cols), 128, 0, s, ma); e->prof_end(s);
            }
        }
    }
    if (lz) {
        Lz4Args za{e->raw.p, e->d_state, e->wire.p, e->comp_size, e->wire_off, e->frame_pfx, e->d_tail, e->frame_bytes, e->lz_phases};
        const size_t smem = lz_smem(e->frame_bytes).total;
        const uint32_t per_sm = (uint32_t)std::max<size_t>(1, std::min<size_t>(LZ_CTAS_PER_SM, (227 * 1024) / (smem + 1024)));
        const uint32_t grid = (uint32_t)std::min<uint64_t>(sz.n_frames_max, (uint64_t)e->sm_count * per_sm);
        join_tail(e);            // the previous batch's checksum kernel still reads the wire bytes and sizes this kernel overwrites
        CK(cudaMemsetAsync(e->frame_pfx, 0, sz.n_frames_max * 8, s));
        // frames are compressed and written at their final wire offset by one kernel (sizes of the earlier frames by decoupled look-back)
        e->prof_begin("k_lz4_frames", s); launch_k_lz4_frames(grid, LZ_THREADS, smem, s, za); e->prof_end(s);
        // the checksum chain (one thread per frame: latency-bound, a few warps per SM) runs on a side stream, under the next batch
        FrameArgs fa{e->comp_size, e->wire_off, e->wire.p, e->d_tail};
        cudaStream_t s3 = e->side2_stream;
        CK(cudaEventRecord(e->ev_fork, s)); CK(cudaStreamWaitEvent(s3, e->ev_fork, 0));
        e->prof_begin("k_frame_seal", s3); launch_k_frame_seal((uint32_t)((sz.n_frames_max + 31) / 32), 32, SEAL_SMEM, s3, fa); e->prof_end(s3);
        CK(cudaEventRecord(e->ev_tail2, s3));
        e->tail_pending = true; e->tail_nrows = n; e->tail_plan = (const void*)&pd; e->tail_nframes_max = sz.n_frames_max;      // joined by whoever needs the wire bytes, or by the next batch before its LZ4
    }
    CK(cudaGetLastError());
}

}  // namespace


// wire format ids accepted by the encode entry points; serializer formats need no sink in the plan
static bool wire_is_ser(int wire_fmt) { const int b = wire_fmt & 0xff; return (b == TF_WIRE_SER_JSON || b == TF_WIRE_SER_CSV) && (wire_fmt & ~(0xff | TF_WIRE_F_CLOSING_NEWLINE | TF_WIRE_F_ANY_AS_STRING)) == 0; }
static bool wire_known(int wire_fmt) { return wire_fmt == TF_WIRE_CH_NATIVE || wire_fmt == TF_WIRE_CH_NATIVE_LZ4 || wire_fmt == TF_WIRE_CH_JSONEACHROW || wire_is_ser(wire_fmt); }

// The plan `plan_id` names, or nullptr for a missing engine or an id out of range (the call answers TF_E_FATAL_ARG).
static PlanDev* plan_arg(tfgpu_engine* e, int plan_id) { return (e && plan_id >= 0 && plan_id < (int)e->plans.size()) ? e->plans[plan_id].get() : nullptr; }
// A wire format the encoder writes, with a sink in the plan unless it is a serializer format; columnar_ok: the parsers' 0 (rows columnar).
static void check_wire(const PlanDev& pd, int wire_fmt, bool columnar_ok) {
    if (columnar_ok && wire_fmt == 0) return;
    if (!wire_known(wire_fmt)) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "wire format not implemented");
    if (!wire_is_ser(wire_fmt) && !pd.plan.has_sink) throw tfplan::FatalError(TF_E_FATAL_CONFIG, "plan was built without a sink");
}
static void check_batch(const PlanDev& pd, const tf_batch* in) {
    if (in->ncols != pd.plan.in_schema.size()) throw tfplan::FatalError(TF_E_FATAL_ARG, "batch column count does not match the plan schema");
    if (in->nrows >= (1ull << 31)) throw tfplan::FatalError(TF_E_FATAL_ARG, "batch too large (>= 2^31 rows)");
}
// Message end offsets of a parser call (end_of(m) = end of message m): non-decreasing, inside the buffer, the last one at its end.
template <class End> static void check_msg_ends(uint64_t len, uint32_t n_msgs, End end_of) {
    uint64_t prev = 0;
    for (uint32_t m = 0; m < n_msgs; m++) {
        const uint64_t end = end_of(m);
        if (end < prev || end > len) throw tfplan::FatalError(TF_E_FATAL_ARG, "message ends must be non-decreasing and inside the buffer");
        prev = end;
    }
    if (prev != len) throw tfplan::FatalError(TF_E_FATAL_ARG, "the messages must cover the whole buffer");
}

extern "C" {

const char* tfgpu_version(void) { return "tfgpu 0.1.0 sm_100a"; }

int tfgpu_engine_create(const char* cfg_json, const int* device_ids, int n_devices, tfgpu_engine** out) {
    if (!out) return TF_E_FATAL_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return TF_E_FATAL_NODEVICE; }
    if (n_devices > 1) return TF_E_FATAL_ARG;
    auto e = std::make_unique<tfgpu_engine>();
    e->device = (n_devices == 1 && device_ids) ? device_ids[0] : 0;
    if (e->device < 0 || e->device >= ndev) return TF_E_FATAL_ARG;
    try {
        if (cfg_json && *cfg_json) {
            auto cfg = tfj::parse(cfg_json);
            double fb = cfg->get_num("frame_bytes", LZ_MAX_FRAME);
            if (fb < 1024 || fb > LZ_MAX_FRAME || ((uint32_t)fb & 15)) return TF_E_FATAL_CONFIG;
            e->frame_bytes = (uint32_t)fb;
        }
        CK(cudaSetDevice(e->device));
        cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, e->device));
        e->sm_count = prop.multiProcessorCount;
        CK(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
        e->stream = e->own_stream;
        CK(cudaStreamCreateWithFlags(&e->side_stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&e->side2_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&e->ev_tail2, cudaEventDisableTiming));
        CK(cudaMalloc(&e->d_tail, 64)); CK(cudaMemset(e->d_tail, 0, 64));
        CK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
        CK(cudaMalloc(&e->d_state, sizeof(DState)));
        CK(lz4_kernels_init()); CK(dbz_kernels_init());
    } catch (const CudaError& c) { return c.e == cudaErrorMemoryAllocation ? TF_E_RETRY_OOM : TF_E_RETRY_LAUNCH; }
    catch (const std::exception&) { return TF_E_FATAL_CONFIG; }
    *out = e.release();
    return TF_OK;
}

int tfgpu_engine_destroy(tfgpu_engine* e) {
    if (!e) return TF_E_FATAL_ARG;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    for (auto& p : e->plans) p->consts.release();
    e->strict_stage.release(); e->lens_arena.release(); e->lens_arena2.release(); e->in_arena.release(); e->work.release(); e->raw.release(); e->slots.release(); e->wire.release(); e->csv_text.release(); e->csv_stage.release(); e->json_msgs.release(); e->n2f_stage.release(); e->n2f_heap.release(); e->off_scratch.release(); e->json_sizes.release();
    if (e->d_state) cudaFree(e->d_state);
    if (e->d_cols) cudaFree(e->d_cols);
    if (e->d_call_slots) { cudaFree(e->d_call_slots); cudaFree(e->d_regions); }
    if (e->pinned) cudaFreeHost(e->pinned);
    if (e->sel_host) cudaFreeHost(e->sel_host);
    if (e->gather_pool) tfgpu_columnar_destroy(e->gather_pool);
    e->sel_stage.release(); e->err_list.release();
    for (auto ev : e->prof_ev) cudaEventDestroy(ev);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    if (e->ev_tail2) cudaEventDestroy(e->ev_tail2);
    if (e->side2_stream) cudaStreamDestroy(e->side2_stream);
    if (e->d_tail) cudaFree(e->d_tail);
    e->dbz_keysz.release(); e->dbz_meta.release(); e->dbz_old.release(); e->dbz_msgsz.release(); e->old_arena.release(); e->part_ids.release();
    if (e->side_stream) cudaStreamDestroy(e->side_stream);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    delete e;
    return TF_OK;
}

const char* tfgpu_last_error(const tfgpu_engine* e) { return e ? e->last_error.c_str() : "null engine"; }
uint64_t tfgpu_engine_launch_count(const tfgpu_engine* e) { return e ? e->launches : 0; }

int tfgpu_profile_enable(tfgpu_engine* e, int on) { if (!e) return TF_E_FATAL_ARG; e->prof_on = on != 0; e->prof_n = 0; return TF_OK; }

const char* tfgpu_profile_read(tfgpu_engine* e) {
    if (!e) return nullptr;
    cudaSetDevice(e->device);
    try { join_tail(e); } catch (const CudaError&) {}
    cudaStreamSynchronize(e->stream);
    std::string j = "[";
    for (int i = 0; i < e->prof_n; i++) {
        float ms = 0; cudaEventElapsedTime(&ms, e->prof_ev[2 * i], e->prof_ev[2 * i + 1]);
        char b[160]; snprintf(b, sizeof b, "%s{\"name\":\"%s\",\"ms\":%.6f}", i ? "," : "", e->prof_names[i], ms); j += b;
    }
    e->prof_json = j + "]";
    return e->prof_json.c_str();
}

int tfgpu_engine_set_stream(tfgpu_engine* e, void* cuda_stream) {
    if (!e) return TF_E_FATAL_ARG;
    if (e->tail_pending) { cudaSetDevice(e->device); cudaStreamSynchronize(e->side_stream); cudaStreamSynchronize(e->side2_stream); e->tail_pending = false; }
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
    return TF_OK;
}

int tfgpu_plan(tfgpu_engine* e, const char* ns, const char* name, const char* schema_json, const char* transformers_json,
               const char* sink_json, int* plan_id) {
    if (!e || !schema_json || !plan_id || !name) return TF_E_FATAL_ARG;
    return guarded(e, [&] {
        auto pd = std::make_unique<PlanDev>();
        pd->plan = tfplan::build_plan(ns ? ns : "", name, schema_json, transformers_json ? transformers_json : "", sink_json ? sink_json : "");
        upload_plan(e, *pd);
        e->plans.push_back(std::move(pd));
        *plan_id = (int)e->plans.size() - 1;
        return TF_OK;
    });
}

// Host-only: build the plan (Suitable / ResultSchema chain, filter grammar, ClickHouse types) without touching a
// device, so a transfer's YAML can be validated where no GPU is present (cmd/trcli validate does the same for the
// reference's transformers: cmd/trcli/config/model.go:57-72).
int tfgpu_plan_validate(const char* ns, const char* name, const char* schema_json, const char* transformers_json,
                        const char* sink_json, char* describe_out, uint64_t cap, char* err_out, uint64_t err_cap) {
    if (!schema_json || !name) return TF_E_FATAL_ARG;
    return validated(describe_out, cap, err_out, err_cap, [&] {
        return tfplan::build_plan(ns ? ns : "", name, schema_json, transformers_json ? transformers_json : "", sink_json ? sink_json : "").describe;
    });
}

const char* tfgpu_plan_describe(tfgpu_engine* e, int plan_id) {
    if (!e || plan_id < 0 || plan_id >= (int)e->plans.size()) return nullptr;
    return e->plans[plan_id]->plan.describe.c_str();
}

static const uint8_t* stage_input(tfgpu_engine* e, const tf_batch* in, std::vector<tf_col>& dev, DevBuf* arena_opt = nullptr);
int tfgpu_push_encode_resident(tfgpu_engine* e, int plan_id, int wire_fmt, const tf_batch* in) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !in) return TF_E_FATAL_ARG;
    return guarded(e, [&] {
        if (!pd->plan.has_sink) return fail(e, TF_E_FATAL_CONFIG, "plan was built without a sink");
        if (in->mem != TF_MEM_DEVICE) return fail(e, TF_E_FATAL_ARG, "tfgpu_push_encode_resident needs a TF_MEM_DEVICE batch");
        check_batch(*pd, in);
        if (wire_fmt != TF_WIRE_CH_NATIVE && wire_fmt != TF_WIRE_CH_NATIVE_LZ4) return fail(e, TF_E_FATAL_UNSUPPORTED, "wire format not implemented");
        std::vector<tf_col> dev; const uint8_t* dev_kinds = stage_input(e, in, dev);    // device pointers pass through; TF_COL_LENS8 / 16 lengths become offsets
        run_chain(e, *pd, in, dev.data(), dev_kinds, wire_fmt);
        return TF_OK;
    });
}

int tfgpu_resident_stats(tfgpu_engine* e, uint64_t* rows_out, uint64_t* raw_bytes, uint64_t* wire_bytes, uint64_t* n_errors) {
    if (!e) return TF_E_FATAL_ARG;
    return guarded(e, [&] {
        join_tail(e);
        DState st; CK(cudaMemcpyAsync(&st, e->d_state, sizeof st, cudaMemcpyDeviceToHost, e->stream)); CK(cudaStreamSynchronize(e->stream));
        if (rows_out) *rows_out = st.n_kept; if (raw_bytes) *raw_bytes = st.raw_total;
        if (wire_bytes) *wire_bytes = e->last_wire_fmt == TF_WIRE_CH_NATIVE_LZ4 ? st.wire_total : st.raw_total;
        if (n_errors) *n_errors = st.n_errors;
        return TF_OK;
    });
}

int tfgpu_resident_fetch(tfgpu_engine* e, int what, uint8_t* dst, uint64_t cap) {
    if (!e || !dst) return TF_E_FATAL_ARG;
    return guarded(e, [&] {
        join_tail(e);
        DState st; CK(cudaMemcpyAsync(&st, e->d_state, sizeof st, cudaMemcpyDeviceToHost, e->stream)); CK(cudaStreamSynchronize(e->stream));
        const bool wire = what == 1 && e->last_wire_fmt == TF_WIRE_CH_NATIVE_LZ4;
        const uint64_t n = wire ? st.wire_total : st.raw_total;
        if (n > cap) return fail(e, TF_E_FATAL_ARG, "destination too small");
        CK(cudaMemcpyAsync(dst, wire ? e->wire.p : e->raw.p, n, cudaMemcpyDeviceToHost, e->stream)); CK(cudaStreamSynchronize(e->stream));
        return TF_OK;
    });
}

static void finish_wire(tfgpu_engine* e, uint64_t n, int wire_fmt, tfgpu_result* r);

int tfgpu_push_encode(tfgpu_engine* e, int plan_id, int wire_fmt, const tf_batch* in, tfgpu_result** out) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !in || !out) return TF_E_FATAL_ARG;
    *out = nullptr;
    return guarded(e, [&] {
        check_wire(*pd, wire_fmt, false);
        check_batch(*pd, in);
        std::vector<tf_col> dev; const uint8_t* dev_kinds = stage_input(e, in, dev);
        run_chain(e, *pd, in, dev.data(), dev_kinds, wire_fmt);
        auto r = std::make_unique<tfgpu_result>();
        finish_wire(e, in->nrows, wire_fmt, r.get());
        *out = r.release();
        return TF_OK;
    });
}

// Two-phase push: only the predicate columns cross PCIe first; k_filter answers with the keep flags; the host gathers the kept rows
// (tfgpu_batch_gather, multi-threaded) and only those go through the whole chain. Same result as tfgpu_push_encode: every transformer is
// row-local, filters keep the rows they kept before, and the rows phase one dropped with an error are reported from phase one.
int tfgpu_push_encode_selective(tfgpu_engine* e, int plan_id, int wire_fmt, const tf_batch* in, int threads, tfgpu_result** out) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !in || !out) return TF_E_FATAL_ARG;
    const tfplan::Plan& pl = pd->plan;
    const uint64_t n = in->nrows; const size_t nc = pl.in_schema.size();
    if (in->mem != TF_MEM_HOST || in->ncols != nc || pd->n_fsteps == 0 || n < 8192 || !wire_known(wire_fmt)) return tfgpu_push_encode(e, plan_id, wire_fmt, in, out);
    std::vector<uint8_t> pred(nc, 0);
    for (const auto& fs : pl.filters) for (const auto& ex : fs.exprs) for (const auto& t : ex) if (t.col >= 0 && (size_t)t.col < nc) pred[t.col] = 1;
    for (size_t c = 0; c < nc; c++) if (pred[c] && in->cols[c].type != pl.in_schema[c].tf) return tfgpu_push_encode(e, plan_id, wire_fmt, in, out);   // loose predicate column: Strictify first, one phase
    *out = nullptr;
    return guarded(e, [&] {
        join_tail(e);
        cudaStream_t s = e->stream;
        static const bool trace = std::getenv("TFGPU_SELECTIVE_TRACE") != nullptr;
        const auto t_0 = std::chrono::steady_clock::now();
        // ---- phase one
        std::vector<tf_col> pc(in->cols, in->cols + nc);
        for (size_t c = 0; c < nc; c++) if (!pred[c]) { pc[c].values = nullptr; pc[c].validity = nullptr; pc[c].offsets = nullptr; pc[c].heap = nullptr; pc[c].aux = nullptr; pc[c].heap_len = 0; pc[c].flags = 0; }
        const tf_batch b1{n, (uint32_t)nc, TF_MEM_HOST, pc.data(), in->kinds};
        std::vector<tf_col> dev; const uint8_t* dev_kinds = stage_input(e, &b1, dev);
        std::vector<DCol> hc(nc);
        for (size_t c = 0; c < nc; c++) hc[c] = plain_dcol(dev[c], pl.in_schema[c].tf);
        if (e->d_cols_cap < nc) { if (e->d_cols) CK(cudaFree(e->d_cols)); CK(cudaMalloc(&e->d_cols, sizeof(DCol) * nc)); e->d_cols_cap = nc; }
        CK(cudaMemcpyAsync(e->d_cols, hc.data(), sizeof(DCol) * nc, cudaMemcpyHostToDevice, s));
        CK(cudaMemsetAsync(e->d_state, 0, sizeof(DState), s));
        const uint32_t nb = (uint32_t)((n + 255) / 256);
        const size_t flags_bytes = align_up(3 * n, 256);
        e->sel_stage.ensure(flags_bytes + (size_t)nb * 4 + 256);
        uint8_t* B = e->sel_stage.p;
        FilterArgs fa{e->d_cols, dev_kinds, n, pd->d_fsteps, pd->n_fsteps, pd->d_expr_off, pd->d_terms, pd->d_blob, B, B + n, B + 2 * n, (uint32_t*)(B + flags_bytes), e->d_state, nullptr, nullptr, 0};
        e->prof_n = 0;
        e->prof_begin("k_filter", s); launch_k_filter(nb, 256, 0, s, fa); e->prof_end(s);
        if (e->sel_host_cap < 3 * n) { if (e->sel_host) CK(cudaFreeHost(e->sel_host)); e->sel_host = nullptr; e->sel_host_cap = 0; const size_t want = align_up(3 * n + 3 * n / 4 + 4096, 1 << 16); CK(cudaMallocHost(&e->sel_host, want)); e->sel_host_cap = want; }
        CK(cudaMemcpyAsync(e->sel_host, B, 3 * n, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        const uint8_t* keep = e->sel_host; const uint8_t* ecode = keep + n; const uint8_t* estep = keep + 2 * n;
        const auto t_1 = std::chrono::steady_clock::now();
        // ---- host gather of the kept rows
        if (!e->gather_pool) { const int rc = tfgpu_columnar_create(&e->gather_pool); if (rc) return fail(e, rc, "cannot create the gather pool"); }
        const tf_batch* kept = nullptr; const uint32_t* sel = nullptr;
        int rc = tfgpu_batch_gather(e->gather_pool, in, keep, threads, &kept, &sel);
        if (rc) return fail(e, rc, std::string("gather: ") + tfgpu_columnar_last_error(e->gather_pool));
        const auto t_2 = std::chrono::steady_clock::now();
        // ---- phase two: the whole chain over the kept rows
        std::vector<tf_col> dev2; const uint8_t* dev_kinds2 = stage_input(e, kept, dev2);
        run_chain(e, *pd, kept, dev2.data(), dev_kinds2, wire_fmt);
        auto r = std::make_unique<tfgpu_result>();
        finish_wire(e, kept->nrows, wire_fmt, r.get());
        r->rows_in = n;
        if (trace) {
            const auto t_3 = std::chrono::steady_clock::now();
            auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
            std::fprintf(stderr, "[tfgpu selective] phase one %.2f ms, gather %.2f ms, phase two %.2f ms (kept %llu of %llu rows)\n", ms(t_0, t_1), ms(t_1, t_2), ms(t_2, t_3), (unsigned long long)kept->nrows, (unsigned long long)n);
        }
        for (auto& er : r->errs) er.row = sel[er.row];
        std::vector<tf_rowerr> first;
        for (uint64_t i = 0; i < n; i++) if (ecode[i]) first.push_back(tf_rowerr{(uint32_t)i, ecode[i], estep[i]});
        if (!first.empty()) {
            first.insert(first.end(), r->errs.begin(), r->errs.end());
            std::sort(first.begin(), first.end(), [](const tf_rowerr& a, const tf_rowerr& b) { return a.row < b.row; });
            r->errs.swap(first);
        }
        *out = r.release();
        return TF_OK;
    });
}
uint64_t tfgpu_engine_h2d_bytes(const tfgpu_engine* e) { return e ? e->h2d_bytes : 0; }

// shared by push_encode / push_columns: stage host columns into HBM (or pass device pointers through)
static const uint8_t* stage_input(tfgpu_engine* e, const tf_batch* in, std::vector<tf_col>& dev, DevBuf* arena_opt) {
    DevBuf& arena = arena_opt ? *arena_opt : e->in_arena;
    DevBuf& larena = arena_opt ? e->lens_arena2 : e->lens_arena;
    // var-width columns that carry lengths instead of offsets (TF_COL_LENS8 / 16): offsets are built on the device
    auto expand_lens = [&](std::vector<tf_col>& dv) {
        const uint64_t nr = in->nrows; std::vector<LensSrc> src; std::vector<uint32_t> which;
        for (uint32_t c = 0; c < in->ncols; c++) if (!in_width(dv[c].type) && (dv[c].flags & (TF_COL_LENS8 | TF_COL_LENS16)) && dv[c].offsets) { src.push_back(LensSrc{(const uint8_t*)dv[c].offsets, (dv[c].flags & TF_COL_LENS8) ? 1 : 2, 0}); which.push_back(c); }
        if (src.empty()) return;
        const size_t K = src.size(), o_src = 0, o_len = align_up(K * sizeof(LensSrc) + 16, 256), o_off = o_len + align_up(K * nr * 4 + 16, 256), o_tot = o_off + align_up(K * (nr + 1) * 4 + 16, 256);
        larena.ensure(o_tot + K * 8 + 256);
        uint8_t* B = larena.p; cudaStream_t st = e->stream;
        CK(cudaMemcpyAsync(B + o_src, src.data(), K * sizeof(LensSrc), cudaMemcpyHostToDevice, st));
        // `src` is pageable: cudaMemcpyAsync has staged it before it returns, so the vector may go out of scope and nothing waits here
        if (nr) { e->launches++; launch_k_widen_lens(dim3((uint32_t)std::min<uint64_t>((nr + 255) / 256, 2048), (uint32_t)K), 256, 0, st, (const LensSrc*)(B + o_src), nr, (uint32_t*)(B + o_len)); }
        launch_offsets(e, (const uint32_t*)(B + o_len), nr, (uint32_t)K, (uint32_t*)(B + o_off), (uint64_t*)(B + o_tot), st);
        for (size_t k = 0; k < K; k++) { dv[which[k]].offsets = (const uint32_t*)(B + o_off) + k * (nr + 1); dv[which[k]].flags &= ~(TF_COL_LENS8 | TF_COL_LENS16); }
    };
    const uint64_t n = in->nrows; const uint32_t nc = in->ncols;
    cudaStream_t s = e->stream;
    dev.resize(nc);
    if (in->mem != TF_MEM_HOST) { for (uint32_t c = 0; c < nc; c++) dev[c] = in->cols[c]; expand_lens(dev); return in->kinds; }
    size_t tot = 0;
    auto sz_of = [&](const tf_col& c, int which) -> size_t {
        const int w = in_width(c.type);
        switch (which) {
        case 0: return w ? (size_t)w * n : 0;
        case 1: return c.validity ? (n + 7) / 8 : 0;
        case 2: return (!w && c.offsets) ? ((c.flags & TF_COL_LENS8) ? n : (c.flags & TF_COL_LENS16) ? 2 * n : (n + 1) * 4) : 0;
        case 3: return (!w) ? c.heap_len : 0;
        default: if (!c.aux) return 0; return (c.type == TF_ANY) ? n : (size_t)4 * n;
        }
    };
    for (uint32_t c = 0; c < nc; c++) for (int k = 0; k < 5; k++) tot += align_up(sz_of(in->cols[c], k) + 16, 256);
    tot += align_up(n + 16, 256);
    arena.ensure(tot);
    uint8_t* p = arena.p;
    // A shim that keeps the whole batch in ONE pinned arena laid out like the device staging (every non-empty buffer at the next multiple of
    // 256 past the previous buffer's end + 16, in the order values / validity / offsets / heap / aux per column, then kinds) gets a single
    // DMA instead of one per buffer: a few hundred descriptors per batch cost several per cent of the PCIe time.
    {
        const uint8_t* first = nullptr; size_t first_off = 0, off = 0, end_off = 0; bool contiguous = true;
        auto chk = [&](const void* src, size_t bytes) {
            if (!src || !bytes) return;
            if (!first) { first = (const uint8_t*)src; first_off = off; }
            else if ((const uint8_t*)src != first + (off - first_off)) contiguous = false;
            end_off = off + bytes; off += align_up(bytes + 16, 256);
        };
        for (uint32_t c = 0; c < nc && contiguous; c++) { const tf_col& ic = in->cols[c]; chk(ic.values, sz_of(ic, 0)); chk(ic.validity, sz_of(ic, 1)); chk(ic.offsets, sz_of(ic, 2)); chk(ic.heap, sz_of(ic, 3)); chk(ic.aux, sz_of(ic, 4)); }
        if (contiguous && in->kinds) chk(in->kinds, n);
        if (contiguous && first && end_off - first_off >= (1u << 20)) {
            CK(cudaMemcpyAsync(p + first_off, first, end_off - first_off, cudaMemcpyHostToDevice, s)); e->h2d_bytes += end_off - first_off;
            auto at = [&](const void* src, size_t bytes) -> uint8_t* { if (!src || !bytes) return nullptr; uint8_t* d = p; p += align_up(bytes + 16, 256); return d; };
            for (uint32_t c = 0; c < nc; c++) {
                const tf_col& ic = in->cols[c]; tf_col& d = dev[c]; d = ic;
                d.values = at(ic.values, sz_of(ic, 0)); d.validity = at(ic.validity, sz_of(ic, 1)); d.offsets = (const uint32_t*)at(ic.offsets, sz_of(ic, 2));
                d.heap = at(ic.heap, sz_of(ic, 3)); if (!in_width(ic.type) && !d.heap) d.heap = arena.p;
                d.aux = at(ic.aux, sz_of(ic, 4));
            }
            const uint8_t* dk1 = in->kinds ? at(in->kinds, n) : nullptr;
            expand_lens(dev);
            return dk1;
        }
    }
    auto up = [&](const void* src, size_t bytes) -> uint8_t* {
        if (!src || !bytes) { return nullptr; }
        uint8_t* d = p; CK(cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, s)); p += align_up(bytes + 16, 256); e->h2d_bytes += bytes; return d;
    };
    for (uint32_t c = 0; c < nc; c++) {
        const tf_col& ic = in->cols[c]; tf_col& d = dev[c]; d = ic;
        d.values = up(ic.values, sz_of(ic, 0)); d.validity = up(ic.validity, sz_of(ic, 1));
        d.offsets = (const uint32_t*)up(ic.offsets, sz_of(ic, 2));
        d.heap = up(ic.heap, sz_of(ic, 3));
        if (!in_width(ic.type) && !d.heap) d.heap = arena.p;   // empty heap: any valid pointer
        d.aux = up(ic.aux, sz_of(ic, 4));
    }
    const uint8_t* dk = in->kinds ? up(in->kinds, n) : nullptr;
    expand_lens(dev);
    return dk;
}

static void fetch_errors(tfgpu_engine* e, uint64_t n, tfgpu_result* r) {
    // only the failing rows come back: (row, code, term) triples collected on the device, sorted by row here
    cudaStream_t s = e->stream;
    DState st; CK(cudaMemcpyAsync(&st, e->d_state, sizeof st, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
    uint64_t cap = std::min<uint64_t>(st.n_errors, n);
    if (!cap) return;
    std::vector<DevRowErr> got;
    for (int attempt = 0; attempt < 2; attempt++) {
        e->err_list.ensure(cap * sizeof(DevRowErr) + 64);
        unsigned long long* counter = (unsigned long long*)e->err_list.p; DevRowErr* list = (DevRowErr*)(e->err_list.p + 16);
        CK(cudaMemsetAsync(counter, 0, 8, s));
        e->launches++; launch_k_collect_errors((uint32_t)((n + 255) / 256), 256, 0, s, e->errcode, e->errstep, n, list, counter, cap);
        got.resize(cap); unsigned long long found = 0;
        CK(cudaMemcpyAsync(got.data(), list, cap * sizeof(DevRowErr), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(&found, counter, 8, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
        if (found <= cap) { got.resize((size_t)found); break; }
        cap = std::min<uint64_t>(found, n);                  // a writer of errcode that did not count its rows: collect again with room for all
    }
    std::sort(got.begin(), got.end(), [](const DevRowErr& a, const DevRowErr& b) { return a.row < b.row; });
    for (const DevRowErr& g : got) r->errs.push_back(tf_rowerr{g.row, g.code, g.term});
}

static void finish_columnar(tfgpu_engine* e, PlanDev& pd, uint64_t n, tfgpu_result* r) {
    cudaStream_t s = e->stream;
    DState st; CK(cudaMemcpyAsync(&st, e->d_state, sizeof st, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
    r->rows_in = n; r->rows_out = st.n_kept; r->raw_len = st.raw_total;
    const size_t no = pd.plan.out_cols.size();
    std::vector<ColRegions> reg(no);
    CK(cudaMemcpyAsync(reg.data(), e->d_regions, sizeof(ColRegions) * no, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    // the returned offsets are uint32: a column of mask digests (64 bytes per row) or of convert_to_string text that passes 4 GiB would wrap
    for (size_t k = 0; k < no; k++) if (reg[k].heap_len >= (1ull << 32))
        throw tfplan::FatalError(TF_E_FATAL_ARG, "push_columns: output column " + std::to_string(k) + " exceeds 4 GiB of text (uint32 offsets); push fewer rows per call");
    uint8_t* buf = (uint8_t*)malloc(st.raw_total ? st.raw_total : 1);
    if (!buf) throw std::bad_alloc();
    r->owned.push_back(buf);
    if (st.raw_total) CK(cudaMemcpyAsync(buf, e->raw.p, st.raw_total, cudaMemcpyDeviceToHost, s));
    if (e->last_has_sharder && st.n_kept) { r->part_ids.resize(st.n_kept); CK(cudaMemcpyAsync(r->part_ids.data(), e->part_ids.p, st.n_kept * 4, cudaMemcpyDeviceToHost, s)); }
    CK(cudaStreamSynchronize(s));
    if (st.n_errors) fetch_errors(e, n, r);
    r->cols.resize(no);
    for (size_t k = 0; k < no; k++) {
        tf_col& c = r->cols[k]; std::memset(&c, 0, sizeof c);
        c.type = pd.plan.out_schema[k].tf;
        auto at = [&](uint64_t off) -> const uint8_t* { return off == ~0ull ? nullptr : buf + off; };
        c.values = at(reg[k].values); c.validity = at(reg[k].validity); c.aux = at(reg[k].aux);
        c.offsets = (const uint32_t*)at(reg[k].offsets); c.heap = at(reg[k].heap); c.heap_len = reg[k].heap_len;
    }
    r->batch.nrows = st.n_kept; r->batch.ncols = (uint32_t)no; r->batch.mem = TF_MEM_HOST; r->batch.cols = r->cols.data(); r->batch.kinds = nullptr;
}

static void finish_wire(tfgpu_engine* e, uint64_t n, int wire_fmt, tfgpu_result* r) {
    cudaStream_t s = e->stream;
    join_tail(e);
    DState st; CK(cudaMemcpyAsync(&st, e->d_state, sizeof st, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
    r->rows_in = n; r->rows_out = st.n_kept; r->raw_len = st.raw_total;
    const bool lz = wire_fmt == TF_WIRE_CH_NATIVE_LZ4;
    r->n_frames = lz ? st.n_frames : 0;
    r->bytes_len = lz ? st.wire_total : st.raw_total;
    if (e->pinned_cap < r->bytes_len + 64) {   // grow-only pinned landing buffer, owned by the engine
        if (e->pinned) { CK(cudaFreeHost(e->pinned)); e->pinned = nullptr; e->pinned_cap = 0; }
        const size_t want = align_up(r->bytes_len + r->bytes_len / 4 + 4096, 1 << 20);
        CK(cudaMallocHost(&e->pinned, want)); e->pinned_cap = want;
    }
    r->bytes = e->pinned; r->bytes_pinned = false;
    CK(cudaMemcpyAsync(r->bytes, lz ? e->wire.p : e->raw.p, r->bytes_len, cudaMemcpyDeviceToHost, s));
    { const int b = wire_fmt & 0xff;
      if ((b == TF_WIRE_SER_JSON || b == TF_WIRE_SER_CSV || b == TF_WIRE_CH_JSONEACHROW || b == TF_WIRE_DEBEZIUM) && st.n_kept) { r->row_sizes.resize(st.n_kept); CK(cudaMemcpyAsync(r->row_sizes.data(), e->json_sizes.p, st.n_kept * 4, cudaMemcpyDeviceToHost, s)); }
      if (b == TF_WIRE_DEBEZIUM && st.n_kept) { r->key_sizes.resize(st.n_kept); CK(cudaMemcpyAsync(r->key_sizes.data(), e->dbz_keysz.p, st.n_kept * 4, cudaMemcpyDeviceToHost, s));
                                                r->msg_sizes.resize(st.n_kept * 7); CK(cudaMemcpyAsync(r->msg_sizes.data(), e->dbz_msgsz.p, st.n_kept * 28, cudaMemcpyDeviceToHost, s)); } }
    if (e->last_has_sharder && st.n_kept) { r->part_ids.resize(st.n_kept); CK(cudaMemcpyAsync(r->part_ids.data(), e->part_ids.p, st.n_kept * 4, cudaMemcpyDeviceToHost, s)); }
    if (st.n_errors) fetch_errors(e, n, r);
    CK(cudaStreamSynchronize(s));
}

// The plan's chain over a parser's device-resident batch: the rows come back columnar (wire_fmt 0) or as wire bytes.
static std::unique_ptr<tfgpu_result> chain_parsed(tfgpu_engine* e, PlanDev& pd, const tf_batch& staged, const uint8_t* kinds, const uint8_t* pre_err, int wire_fmt) {
    run_chain(e, pd, &staged, staged.cols, kinds, wire_fmt == 0 ? TF_WIRE_COLUMNAR_INTERNAL : wire_fmt, pre_err);
    auto r = std::make_unique<tfgpu_result>();
    if (wire_fmt == 0) finish_columnar(e, pd, staged.nrows, r.get()); else finish_wire(e, staged.nrows, wire_fmt, r.get());
    return r;
}

// TransformerResult{Transformed, Errors}: the kept rows come back columnar in host memory owned by the result.
int tfgpu_push_columns(tfgpu_engine* e, int plan_id, const tf_batch* in, tfgpu_result** out) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !in || !out) return TF_E_FATAL_ARG;
    *out = nullptr;
    return guarded(e, [&] {
        check_batch(*pd, in);
        std::vector<tf_col> dev; const uint8_t* dev_kinds = stage_input(e, in, dev);
        run_chain(e, *pd, in, dev.data(), dev_kinds, TF_WIRE_COLUMNAR_INTERNAL);
        auto r = std::make_unique<tfgpu_result>();
        finish_columnar(e, *pd, in->nrows, r.get());
        *out = r.release();
        return TF_OK;
    });
}

// Queue Debezium serializer for columns without a database-specific original_type (Emitter.EmitKV
// pkg/debezium/emitter_value_converter.go:626-690). The per-table constants become a text template once per (plan, opts).
namespace {
__global__ void k_dbz_kinds(const uint8_t* kinds, uint64_t n, uint8_t* pre_err) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) pre_err[r] = kinds[r] == TF_KIND_INSERT ? 0 : TF_ROWERR_DBZ_EMIT_HOST;
}
// Host part of the emitter set-up, independent of any device state (tfgpu_emit_debezium_validate exports it for tests without a GPU):
// the AddPg / addCommon branch of every result column and the message template.
struct DbzHostTpl { std::vector<int> forms; std::string text; std::vector<DbzSeg> segs; };
DbzHostTpl dbz_host_template(const tfplan::Plan& pl, const std::string& opts_json) {
    auto ov = tfj::parse(opts_json);

    // per result column: addCommon, or the AddPg branch (pkg/debezium/pg/emitter.go:265-629) its (original type, column type) pair takes
    std::vector<int> forms(pl.out_schema.size(), DF_COMMON); bool any_common = false;
    for (size_t k = 0; k < pl.out_schema.size(); k++) {
        const tfplan::ColSchema& c = pl.out_schema[k]; const std::string& ot = c.original_type;
        const bool typed = ot.rfind("pg:", 0) == 0 || ot.rfind("mysql:", 0) == 0 || ot.rfind("ydb:", 0) == 0;
        if (!typed) { any_common = true; continue; }
        int f = -1;
        bool untouched = !(pl.tostr_col.size() > (size_t)c.in_index && pl.tostr_col[(size_t)c.in_index]) && !(pl.todt_col.size() > (size_t)c.in_index && pl.todt_col[(size_t)c.in_index]);
        for (auto& ms : pl.masks) for (int mc : ms.cols) if (mc == c.in_index) untouched = false;
        auto is = [&](const char* t) { return ot == t; };
        static const std::regex re_char("pg:character( varying)?(\\([0-9]+\\))?"), re_ts("pg:timestamp(\\(([0-9])\\))? without time zone"), re_tstz("pg:timestamp(\\([0-6]\\))? with time zone");
        std::smatch m;
        if (is("pg:boolean")) f = c.tf == TF_BOOLEAN ? DF_COMMON : -1;
        else if (is("pg:smallint")) f = c.tf == TF_INT16 ? DF_COMMON : -1;
        else if (is("pg:integer")) f = c.tf == TF_INT32 ? DF_COMMON : -1;
        else if (is("pg:bigint")) f = c.tf == TF_INT64 ? DF_COMMON : -1;
        else if (is("pg:bytea")) f = c.tf == TF_BYTES ? DF_COMMON : -1;
        else if (is("pg:real")) f = (c.tf == TF_DOUBLE || c.tf == TF_FLOAT) ? DF_PG_REAL : -1;
        else if (is("pg:double precision")) f = c.tf == TF_DOUBLE ? DF_PG_DOUBLE : -1;
        else if (is("pg:text") || is("pg:uuid") || is("pg:cidr") || is("pg:macaddr") || is("pg:citext") || is("pg:int4range") || is("pg:int8range") || std::regex_match(ot, re_char))
            f = (c.tf == TF_UTF8 || c.tf == TF_ANY) ? DF_PG_STRING : -1;
        else if (is("pg:json") || is("pg:jsonb")) f = c.tf == TF_ANY ? DF_PG_JSON : -1;
        else if (is("pg:inet")) f = (c.tf == TF_UTF8 || c.tf == TF_ANY) ? DF_PG_INET : -1;
        else if (is("pg:date")) f = c.tf == TF_DATE ? DF_PG_DATE : -1;
        else if (std::regex_match(ot, m, re_ts)) f = c.tf != TF_TIMESTAMP ? -1 : (m[2].matched && m[2].str()[0] >= '1' && m[2].str()[0] <= '3') ? DF_PG_TS_MILLIS : DF_PG_TS_MICROS;   // GetTimeDivider typeutil/helpers.go:104-120
        else if (std::regex_match(ot, re_tstz)) f = c.tf == TF_TIMESTAMP ? DF_PG_TSTZ : -1;
        if (f < 0 || !untouched)
            throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "column " + c.name + ": original_type " + ot + " (column type " + c.type + ") is emitted by the database-specific converters of the Go emitter");
        forms[k] = f;
    }
    if (any_common && !ov->get_bool("ignore_unknown_sources"))
        throw tfplan::FatalError(TF_E_FATAL_CONFIG, "unknown source type (emitter_value_converter.go:183-191): a column has no original_type; set ignore_unknown_sources");
    const bool snapshot = ov->get_bool("snapshot"), drop_keys = ov->get_bool("drop_keys");
    const std::string st = ov->get_str("source_type");
    if (!(st.empty() || st == "pg" || st == "mysql")) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "source_type " + st);
    auto q = [](const std::string& t) { return host_json_quote_nohtml(t); };
    auto wrap = [&](const char* schema_key, const char* id_key, std::string& prefix, std::string& suffix) {
        const tfj::Value* idv = ov->get(id_key); const tfj::Value* sv = ov->get(schema_key);
        if (idv && idv->kind == tfj::Value::Num) {                                   // packer_schema_registry.go:66-76
            const uint32_t id = (uint32_t)idv->num; prefix.push_back('\0'); for (int sh = 24; sh >= 0; sh -= 8) prefix.push_back((char)((id >> sh) & 0xff));
        } else if (sv && sv->kind == tfj::Value::Str) { prefix = "{\"payload\":"; suffix = ",\"schema\":" + sv->str + "}"; }     // packer_include_schema.go:34-38
    };
    std::string text; std::vector<DbzSeg> segs;
    auto seg = [&](const std::string& t, int code) { segs.push_back(DbzSeg{(int32_t)text.size(), (int32_t)t.size(), code, 0}); text += t; };
    if (drop_keys) seg("", DZ_KEY_END);
    else { std::string pre, suf; wrap("key_schema", "key_schema_id", pre, suf); seg(pre, DZ_KEY); seg(suf, DZ_KEY_END); }
    std::string pre, suf; wrap("val_schema", "val_schema_id", pre, suf);
    seg(pre + "{\"after\":", DZ_AFTER);
    seg(",\"before\":", DZ_BEFORE);                                                  // null, or OldKeys for update (replica identity full) / delete events
    seg(",\"op\":\"", DZ_OP);                                                        // kindToOp kind.go:8-31
    const std::string name = q(ov->get_str("topic_prefix")), db = q(ov->get_str("database")), ver = q(ov->get_str("version"));
    const std::string snap = snapshot ? "\"true\"" : "\"false\"", tbl = q(pl.out_name), sch = q(pl.out_ns);
    const std::string head = "\",\"source\":{";
    if (st == "pg") {                 // buildSource :329-372, keys in encoding/json's sorted order
        seg(head + "\"connector\":\"postgresql\",\"db\":" + db + ",\"lsn\":", DZ_LSN);
        seg(",\"name\":" + name + ",\"schema\":" + sch + ",\"snapshot\":" + snap + ",\"table\":" + tbl + ",\"ts_ms\":", DZ_SRC_TS);
        seg(",\"txId\":", DZ_ID);
        seg(",\"version\":" + ver + ",\"xmin\":null},\"transaction\":null,\"ts_ms\":", DZ_TS);
    } else if (st == "mysql") {
        seg(head + "\"connector\":\"mysql\",\"db\":" + sch + ",\"file\":\"mysql-log.", DZ_FILE);
        seg("\",\"gtid\":", DZ_GTID);
        seg(",\"name\":" + name + ",\"pos\":", DZ_POS);
        seg(",\"query\":null,\"row\":0,\"server_id\":0,\"snapshot\":" + snap + ",\"table\":" + tbl + ",\"thread\":null,\"ts_ms\":", DZ_SRC_TS);
        seg(",\"version\":" + ver + "},\"transaction\":null,\"ts_ms\":", DZ_TS);
    } else {
        seg(head + "\"db\":" + db + ",\"name\":" + name + ",\"snapshot\":" + snap + ",\"table\":" + tbl + ",\"ts_ms\":", DZ_SRC_TS);
        seg(",\"version\":" + ver + "},\"transaction\":null,\"ts_ms\":", DZ_TS);
    }
    seg("}" + suf, DZ_NONE);
    DbzHostTpl t; t.forms = std::move(forms); t.text = std::move(text); t.segs = std::move(segs);
    return t;
}

void dbz_build_template(PlanDev& pd, const std::string& opts_json) {
    if (pd.dbz_opts_key == opts_json && pd.dbz.segs) return;
    const tfplan::Plan& pl = pd.plan;
    const DbzHostTpl ht = dbz_host_template(pl, opts_json);
    const std::vector<int>& forms = ht.forms; const std::string& text = ht.text; const std::vector<DbzSeg>& segs = ht.segs;
    std::vector<JsonCol> acols = pd.h_sjcols, kcols;
    for (JsonCol& jc : acols) jc.pad1 = forms[(size_t)jc.pad0];
    for (const JsonCol& jc : acols) if (pl.out_schema[(size_t)jc.pad0].key) kcols.push_back(jc);
    const size_t o_seg = 0, o_text = align_up(segs.size() * sizeof(DbzSeg), 256), o_k = o_text + align_up(text.size() + 1, 256), o_a = o_k + align_up(kcols.size() * sizeof(JsonCol) + 1, 256);
    pd.dbz_consts.ensure(o_a + acols.size() * sizeof(JsonCol) + 256);
    if (!acols.empty()) CK(cudaMemcpy(pd.dbz_consts.p + o_a, acols.data(), acols.size() * sizeof(JsonCol), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(pd.dbz_consts.p + o_seg, segs.data(), segs.size() * sizeof(DbzSeg), cudaMemcpyHostToDevice));
    if (!text.empty()) CK(cudaMemcpy(pd.dbz_consts.p + o_text, text.data(), text.size(), cudaMemcpyHostToDevice));
    if (!kcols.empty()) CK(cudaMemcpy(pd.dbz_consts.p + o_k, kcols.data(), kcols.size() * sizeof(JsonCol), cudaMemcpyHostToDevice));
    pd.dbz = DbzEmitArgs{}; pd.dbz.segs = (const DbzSeg*)(pd.dbz_consts.p + o_seg); pd.dbz.nseg = (int)segs.size(); pd.dbz.text = pd.dbz_consts.p + o_text;
    pd.dbz.kcols = (const JsonCol*)(pd.dbz_consts.p + o_k); pd.dbz.nkc = (int)kcols.size(); pd.dbz.acols = (const JsonCol*)(pd.dbz_consts.p + o_a);
    pd.dbz_opts_key = opts_json;
}
}  // namespace

// Host-only: what tfgpu_emit_debezium would set up for this table and opts_json (no GPU needed). describe_out receives
// {"forms":[per result column],"keys":[result column indexes in key-message order],"template":[[text, code], ...]}.
int tfgpu_emit_debezium_validate(const char* ns, const char* name, const char* schema_json, const char* transformers_json, const char* opts_json,
                                 char* describe_out, uint64_t cap, char* err_out, uint64_t err_cap) {
    if (!schema_json || !name || !opts_json) return TF_E_FATAL_ARG;
    return validated(describe_out, cap, err_out, err_cap, [&] {
        const tfplan::Plan pl = tfplan::build_plan(ns ? ns : "", name, schema_json, transformers_json ? transformers_json : "", "");
        const DbzHostTpl t = dbz_host_template(pl, opts_json);
        std::vector<size_t> order(pl.out_schema.size()); for (size_t k = 0; k < order.size(); k++) order[k] = k;
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return pl.out_schema[a].name < pl.out_schema[b].name; });
        std::string d = "{\"forms\":[";
        for (size_t k = 0; k < t.forms.size(); k++) { if (k) d += ","; d += std::to_string(t.forms[k]); }
        d += "],\"keys\":["; bool first = true;
        for (size_t k : order) if (pl.out_schema[k].key) { if (!first) d += ","; first = false; d += std::to_string(k); }
        d += "],\"template\":[";
        for (size_t g = 0; g < t.segs.size(); g++) {
            if (g) d += ",";
            d += "[" + host_json_quote_nohtml(t.text.substr((size_t)t.segs[g].text_off, (size_t)t.segs[g].text_len)) + "," + std::to_string(t.segs[g].code) + "]";
        }
        return d + "]}";
    });
}

int tfgpu_emit_debezium(tfgpu_engine* e, int plan_id, const char* opts_json, const tf_batch* in, const tf_row_meta* meta, tfgpu_result** out) {
    return tfgpu_emit_debezium_crud(e, plan_id, opts_json, in, nullptr, meta, out);
}

int tfgpu_emit_debezium_crud(tfgpu_engine* e, int plan_id, const char* opts_json, const tf_batch* in, const tf_old_keys* old, const tf_row_meta* meta, tfgpu_result** out) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !in || !out || !opts_json) return TF_E_FATAL_ARG;
    *out = nullptr;
    return guarded(e, [&] {
        check_batch(*pd, in);
        const uint64_t n = in->nrows;
        cudaStream_t s = e->stream;
        try { dbz_build_template(*pd, opts_json); } catch (const std::runtime_error& x) { throw tfplan::FatalError(TF_E_FATAL_CONFIG, std::string("opts_json: ") + x.what()); }
        std::vector<tf_col> dev; const uint8_t* dev_kinds = stage_input(e, in, dev);
        e->dbz = pd->dbz;
        const size_t o_id = 0, o_lsn = align_up(n * 4 + 16, 256), o_ct = o_lsn + align_up(n * 8 + 16, 256), o_off = o_ct + align_up(n * 8 + 16, 256), o_pre = o_off + align_up((n + 1) * 4 + 16, 256), o_heap = o_pre + align_up(n + 16, 256);
        uint64_t gt_len = 0;
        if (meta && in->mem == TF_MEM_HOST && meta->txid_offsets && meta->txid_heap) gt_len = meta->txid_offsets[n];
        e->dbz_meta.ensure(o_heap + gt_len + 256);
        uint8_t* M = e->dbz_meta.p;
        if (meta) {
            if (in->mem == TF_MEM_HOST) {
                if (meta->id && n) { CK(cudaMemcpyAsync(M + o_id, meta->id, n * 4, cudaMemcpyHostToDevice, s)); e->dbz.id = (const uint32_t*)(M + o_id); }
                if (meta->lsn && n) { CK(cudaMemcpyAsync(M + o_lsn, meta->lsn, n * 8, cudaMemcpyHostToDevice, s)); e->dbz.lsn = (const uint64_t*)(M + o_lsn); }
                if (meta->commit_time && n) { CK(cudaMemcpyAsync(M + o_ct, meta->commit_time, n * 8, cudaMemcpyHostToDevice, s)); e->dbz.ct = (const uint64_t*)(M + o_ct); }
                if (meta->txid_offsets && meta->txid_heap && n) {
                    CK(cudaMemcpyAsync(M + o_off, meta->txid_offsets, (n + 1) * 4, cudaMemcpyHostToDevice, s)); e->dbz.gt_off = (const uint32_t*)(M + o_off);
                    if (gt_len) CK(cudaMemcpyAsync(M + o_heap, meta->txid_heap, gt_len, cudaMemcpyHostToDevice, s));
                    e->dbz.gt_heap = M + o_heap;
                }
            } else { e->dbz.id = meta->id; e->dbz.lsn = meta->lsn; e->dbz.ct = meta->commit_time; e->dbz.gt_off = meta->txid_offsets; e->dbz.gt_heap = meta->txid_heap; }
        }
        // update / delete events: kinds + OldKeys (as a second set of typed columns) reach the row writer
        {
            auto ov = tfj::parse(opts_json);
            const tfplan::Plan& pl = pd->plan; const size_t nc = pl.in_schema.size();
            e->dbz.kinds = dev_kinds; e->dbz.snapshot = ov->get_bool("snapshot") ? 1 : 0; e->dbz.mysql_src = ov->get_str("source_type") == "mysql" ? 1 : 0;
            const tfj::Value* tv = ov->get("tombstones_on_delete"); e->dbz.tombstones = (tv && tv->kind == tfj::Value::Bool && !tv->b) ? 0 : 1;      // tombstones.on.delete, default true
            int npk = 0; for (const auto& c : pl.out_schema) if (c.key) npk++;
            e->dbz.n_pkeys = npk; e->dbz.old_cols = nullptr; e->dbz.old_present = nullptr; e->dbz.old_has = nullptr; e->dbz.n_old_present = 0;
            if (old && old->values) {
                if (old->values->ncols != nc || old->values->nrows != n || old->values->mem != in->mem) return fail(e, TF_E_FATAL_ARG, "old keys: same shape and memory space as the batch expected");
                if (!pl.masks.empty() || !pl.todt_cols.empty() || !pl.tostr_cols.empty() || !pl.n2f_cols.empty()) return fail(e, TF_E_FATAL_UNSUPPORTED, "update / delete events after a transformer that rewrites values are emitted by the Go emitter");
                std::vector<tf_col> odev; stage_input(e, old->values, odev, &e->old_arena);
                std::vector<DCol> oc(nc); std::vector<uint8_t> present(nc, 0); int np = 0;
                for (size_t c = 0; c < nc; c++) {
                    const tf_col& ic = odev[c];
                    if (ic.type != pl.in_schema[c].tf) return fail(e, TF_E_FATAL_ARG, "old keys: column " + std::to_string(c) + " type does not match the plan schema");
                    DCol& d = oc[c]; d = plain_dcol(ic, ic.type); d.out_kind = OK_COPY; d.out_w = d.in_w;
                    present[c] = (old->present_cols && old->present_cols[c]) ? 1 : 0; np += present[c];
                    if (present[c] && n) { if (d.in_w && !d.values) return fail(e, TF_E_FATAL_ARG, "old keys: values pointer is NULL"); if (!d.in_w && !d.offsets) return fail(e, TF_E_FATAL_ARG, "old keys: offsets pointer is NULL"); }
                }
                const size_t o_oc = 0, o_pr = align_up(nc * sizeof(DCol) + 16, 256), o_has = o_pr + align_up(nc + 16, 256);
                e->dbz_old.ensure(o_has + n + 256);
                CK(cudaMemcpyAsync(e->dbz_old.p + o_oc, oc.data(), nc * sizeof(DCol), cudaMemcpyHostToDevice, s));
                CK(cudaMemcpyAsync(e->dbz_old.p + o_pr, present.data(), nc, cudaMemcpyHostToDevice, s));
                e->dbz.old_cols = (const DCol*)(e->dbz_old.p + o_oc); e->dbz.old_present = e->dbz_old.p + o_pr; e->dbz.n_old_present = np;
                if (old->row_has && n) {
                    if (in->mem == TF_MEM_HOST) { CK(cudaMemcpyAsync(e->dbz_old.p + o_has, old->row_has, n, cudaMemcpyHostToDevice, s)); e->dbz.old_has = e->dbz_old.p + o_has; }
                    else e->dbz.old_has = old->row_has;
                }
                CK(cudaStreamSynchronize(s));      // oc / present are stack vectors
            }
        }
        run_chain(e, *pd, in, dev.data(), dev_kinds, TF_WIRE_DEBEZIUM, nullptr);
        auto r = std::make_unique<tfgpu_result>();
        finish_wire(e, n, TF_WIRE_DEBEZIUM, r.get());
        *out = r.release();
        return TF_OK;
    });
}

// Measurer middleware (synchronizer/measurer.go:38-42): Size.Values of every row and their sum, in one pass over the columns.
int tfgpu_measure(tfgpu_engine* e, const tf_batch* in, uint64_t* per_row, uint64_t* total) {
    if (!e || !in || !total) return TF_E_FATAL_ARG;
    return guarded(e, [&] {
        cudaStream_t s = e->stream;
        join_tail(e);                     // the work arena is reused below
        std::vector<tf_col> dev; stage_input(e, in, dev);
        const size_t nc = in->ncols; const uint64_t n = in->nrows;
        if (e->d_cols_cap < nc) { if (e->d_cols) CK(cudaFree(e->d_cols)); CK(cudaMalloc(&e->d_cols, sizeof(DCol) * (nc ? nc : 1))); e->d_cols_cap = nc; }
        std::vector<DCol> hc(nc);
        for (size_t c = 0; c < nc; c++) hc[c] = plain_dcol(dev[c], dev[c].type);
        e->work.ensure(n * 8 + 256);
        unsigned long long* d_total = (unsigned long long*)e->work.p; uint64_t* d_rows = per_row ? (uint64_t*)(e->work.p + 64) : nullptr;
        CK(cudaMemcpyAsync(e->d_cols, hc.data(), sizeof(DCol) * nc, cudaMemcpyHostToDevice, s));
        CK(cudaMemsetAsync(d_total, 0, 8, s));
        e->prof_n = 0;
        if (n) { MeasureArgs ma{e->d_cols, (int)nc, n, d_rows, d_total}; e->prof_begin("k_measure", s); launch_k_measure((uint32_t)((n + 255) / 256), 256, 0, s, ma); e->prof_end(s); CK(cudaGetLastError()); }
        CK(cudaMemcpyAsync(total, d_total, 8, cudaMemcpyDeviceToHost, s));
        if (per_row && n) CK(cudaMemcpyAsync(per_row, d_rows, n * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return TF_OK;
    });
}

// ---------------------------------------------------------------------------------------------- CSV
// parsers.Parser for the S3 CSV source (pkg/providers/s3/reader/registry/csv/reader_csv.go:85-452) fused with the
// transformer chain and, when wire_fmt != 0, the ClickHouse encode: raw bytes in, Transformed rows or wire bytes out.
namespace {
struct CsvHostOpts { CsvCfg cfg; std::vector<uint8_t> blob; uint64_t skip = 0; };

uint32_t put_list(std::vector<uint8_t>& blob, const std::vector<std::string>& v) {
    if (v.empty()) return 0xffffffffu;
    while (blob.size() % 4) blob.push_back(0);
    const uint32_t at = (uint32_t)blob.size();
    std::vector<uint32_t> hdr; hdr.push_back((uint32_t)v.size()); uint32_t o = 0; hdr.push_back(0);
    for (auto& x : v) { o += (uint32_t)x.size(); hdr.push_back(o); }
    const uint8_t* h = (const uint8_t*)hdr.data(); blob.insert(blob.end(), h, h + hdr.size() * 4);
    for (auto& x : v) blob.insert(blob.end(), x.begin(), x.end());
    return at;
}

CsvHostOpts parse_csv_opts(const char* js) {
    CsvHostOpts h; std::memset(&h.cfg, 0, sizeof h.cfg);
    h.cfg.delimiter = ','; h.cfg.quote = '"'; h.cfg.escape = '\\'; h.cfg.double_quote = 1;
    std::vector<std::string> nulls, trues, falses;
    if (js && *js) {
        auto v = tfj::parse(js);
        auto ch = [&](const char* k, uint8_t def) -> uint8_t { const tfj::Value* x = v->get(k); if (!x) return def; if (x->kind == tfj::Value::Str) return x->str.empty() ? 0 : (uint8_t)x->str[0]; return def; };
        h.cfg.delimiter = ch("delimiter", ','); h.cfg.quote = ch("quote", '"'); h.cfg.escape = ch("escape", '\\');
        h.cfg.double_quote = v->get_bool("double_quote", true); h.cfg.strings_can_be_null = v->get_bool("strings_can_be_null");
        h.cfg.quoted_strings_can_be_null = v->get_bool("quoted_strings_can_be_null"); h.cfg.include_missing = v->get_bool("include_missing_columns");
        nulls = v->get_str_list("null_values"); trues = v->get_str_list("true_values"); falses = v->get_str_list("false_values");
        h.skip = (uint64_t)v->get_num("skip_lines", 0);
    }
    if (!h.cfg.delimiter || h.cfg.delimiter == '\r' || h.cfg.delimiter == '\n' || h.cfg.delimiter >= 0x80)
        throw tfplan::FatalError(TF_E_FATAL_CONFIG, "csv: invalid delimiter (reader.go:320-322; the device handles ASCII delimiters)");
    if (h.cfg.quote >= 0x80 || h.cfg.escape >= 0x80) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "csv: non-ASCII quote / escape characters");
    h.blob.resize(4, 0);
    h.cfg.null_list = put_list(h.blob, nulls); h.cfg.true_list = put_list(h.blob, trues); h.cfg.false_list = put_list(h.blob, falses);
    return h;
}
}  // namespace

int tfgpu_parse_csv(tfgpu_engine* e, int plan_id, const char* opts_json, const uint8_t* bytes, uint64_t len, int mem, int wire_fmt, tfgpu_result** out) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !out || (!bytes && len)) return TF_E_FATAL_ARG;
    *out = nullptr;
    return guarded(e, [&] {
        if (len >= (1ull << 32) - 16) throw tfplan::FatalError(TF_E_FATAL_ARG, "csv chunk must be < 4 GiB (line positions are uint32)");
        check_wire(*pd, wire_fmt, true);
        cudaStream_t s = e->stream;
        CsvHostOpts ho = parse_csv_opts(opts_json);
        const tfplan::Plan& pl = pd->plan; const size_t nc = pl.in_schema.size();
        // text into HBM
        const uint8_t* d_text = bytes;
        if (mem == TF_MEM_HOST) { e->csv_text.ensure(len + 64); if (len) CK(cudaMemcpyAsync(e->csv_text.p, bytes, len, cudaMemcpyHostToDevice, s)); d_text = e->csv_text.p; }
        // newline index
        const uint32_t nblk = (uint32_t)((len + CSV_NL_BLOCK - 1) / CSV_NL_BLOCK);
        uint64_t nlines = 0;
        e->work.ensure(((size_t)nblk * 8 + 1024) * 2 + 4096);
        uint32_t* blk_cnt = (uint32_t*)e->work.p; uint32_t* blk_off = blk_cnt + align_up(nblk + 1, 64);
        if (nblk) {
            CK(cudaMemsetAsync(e->d_state, 0, sizeof(DState), s));
            e->prof_n = 0;
            e->prof_begin("k_csv_count_nl", s); launch_k_csv_count_nl(nblk, 256, 0, s, d_text, len, blk_cnt, nullptr); e->prof_end(s);
            e->prof_begin("k_scan_blockcnt", s); launch_k_scan_blockcnt(1, 1024, 0, s, blk_cnt, blk_off, nblk, e->d_state); e->prof_end(s);
            DState st; CK(cudaMemcpyAsync(&st, e->d_state, sizeof st, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
            nlines = st.n_kept;
        }
        const uint64_t skip = ho.skip < nlines ? ho.skip : nlines;
        const uint64_t nrows = nlines - skip;
        // staging layout
        std::vector<CsvColDev> hc(nc); std::vector<int16_t> next_same(nc, -1); int nfields = 0, nslots = 0;
        for (size_t c = 0; c < nc; c++) {
            const tfplan::ColSchema& cs = pl.in_schema[c]; CsvColDev& d = hc[c]; std::memset(&d, 0, sizeof d);
            d.tf = cs.tf; d.w = in_width(cs.tf); d.slot = -1;
            d.path = cs.path.empty() ? (int)c : atoi(cs.path.c_str());        // reader_csv.go:286 strconv.Atoi(col.Path)
            if (!cs.path.empty() && cs.path.find_first_not_of("-0123456789") != std::string::npos) throw tfplan::FatalError(TF_E_FATAL_CONFIG, "csv: column path '" + cs.path + "' is not an index");
            if (d.path >= 0 && d.path + 1 > nfields) nfields = d.path + 1;
            if (!d.w) d.slot = nslots++;
        }
        if (nfields > 32000) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "csv: too many fields");
        std::vector<int16_t> field_col(nfields ? nfields : 1, -1);
        for (int c = (int)nc - 1; c >= 0; c--) if (hc[c].path >= 0) { next_same[c] = field_col[hc[c].path]; field_col[hc[c].path] = (int16_t)c; }
        ArenaLayout need;
        const size_t o_line = need((nlines + 1) * 4), o_err = need(nrows), o_cols = need(nc * sizeof(CsvColDev)), o_fc = need(field_col.size() * 2), o_ns = need(nc * 2),
                     o_blob = need(ho.blob.size()), o_ss = need((size_t)nslots * nrows * 4), o_sl = need((size_t)nslots * nrows * 4),
                     o_off = need((size_t)nslots * (nrows + 1) * 4), o_tot = need((size_t)nslots * 8 + 8), o_base = need((size_t)nslots * 8 + 8);
        std::vector<size_t> o_val(nc), o_aux(nc);
        for (size_t c = 0; c < nc; c++) {
            o_val[c] = hc[c].w ? need((size_t)hc[c].w * nrows) : 0;
            const int tf = hc[c].tf;
            o_aux[c] = (tf == TF_DATE || tf == TF_DATETIME || tf == TF_TIMESTAMP) ? need(4 * nrows) : (tf == TF_ANY ? need(nrows) : 0);
        }
        e->csv_stage.ensure(need.total + 256);
        uint8_t* B = e->csv_stage.p;
        for (size_t c = 0; c < nc; c++) {
            if (hc[c].w) hc[c].values = B + o_val[c];
            const int tf = hc[c].tf;
            if (tf == TF_DATE || tf == TF_DATETIME || tf == TF_TIMESTAMP) hc[c].aux32 = (uint32_t*)(B + o_aux[c]);
            if (tf == TF_ANY) hc[c].aux8 = B + o_aux[c];
        }
        CK(cudaMemcpyAsync(B + o_cols, hc.data(), nc * sizeof(CsvColDev), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(B + o_fc, field_col.data(), field_col.size() * 2, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(B + o_ns, next_same.data(), nc * 2, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(B + o_blob, ho.blob.data(), ho.blob.size(), cudaMemcpyHostToDevice, s));
        VarHeaps heaps(nslots);
        if (nlines) { e->prof_begin("k_csv_line_index", s); launch_k_csv_line_index(nblk, 256, 0, s, d_text, len, blk_off, (uint32_t*)(B + o_line), nullptr); e->prof_end(s); }
        if (nrows) {
            CsvArgs ca{d_text, len, (const uint32_t*)(B + o_line), nlines, skip, ho.cfg, B + o_blob, (const CsvColDev*)(B + o_cols), (int)nc,
                       (const int16_t*)(B + o_fc), nfields, (const int16_t*)(B + o_ns), (uint32_t*)(B + o_ss), (uint32_t*)(B + o_sl), B + o_err};
            e->prof_begin("k_csv_pass1", s); launch_k_csv_pass1((uint32_t)std::min<uint64_t>((nrows + CSV_TILE_ROWS - 1) / CSV_TILE_ROWS, (uint64_t)e->sm_count * 16), 32 * CSV_WARPS, 0, s, ca); e->prof_end(s);
            if (nslots) {
                place_heaps(e, heaps, (const uint32_t*)(B + o_sl), nrows, nslots, (uint32_t*)(B + o_off), (uint64_t*)(B + o_tot), (uint64_t*)(B + o_base), "csv chunk");
                CsvCopyArgs cp{d_text, (const uint32_t*)(B + o_ss), (const uint32_t*)(B + o_sl), (const uint32_t*)(B + o_off), heaps.heap, (const uint64_t*)(B + o_base), nrows};
                e->prof_begin("k_csv_pass2", s); launch_k_csv_pass2(dim3((uint32_t)((nrows + 255) / 256), nslots), 256, 0, s, cp); e->prof_end(s);
            }
        }
        std::vector<tf_col> dev;
        auto r = chain_parsed(e, *pd, parsed_batch(hc, nrows, (const uint32_t*)(B + o_off), heaps, dev), nullptr, nrows ? B + o_err : nullptr, wire_fmt);
        uint32_t last_end = 0;
        if (nlines) { CK(cudaMemcpyAsync(&last_end, (uint32_t*)(B + o_line) + (nlines - 1), 4, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s)); }
        r->consumed = last_end;
        *out = r.release();
        return TF_OK;
    });
}

// ---------------------------------------------------------------------------------------------- JSON lines
// parsers.Parser.DoBatch of the generic JSON parser (pkg/parsers/generic/generic_parser.go:406-430,519-555) fused with the
// transformer chain and the sink encode: message bytes in, Transformed rows or wire bytes out.
int tfgpu_parse_json(tfgpu_engine* e, int plan_id, const char* opts_json, const uint8_t* bytes, uint64_t len, int mem,
                     const tf_msg* msgs, uint32_t n_msgs, int wire_fmt, tfgpu_result** out) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !out || (!bytes && len) || (!msgs && n_msgs)) return TF_E_FATAL_ARG;
    *out = nullptr;
    return guarded(e, [&] {
        if (len >= (1ull << 32) - 16) throw tfplan::FatalError(TF_E_FATAL_ARG, "json batch must be < 4 GiB (line positions are uint32)");
        check_wire(*pd, wire_fmt, true);
        check_msg_ends(len, n_msgs, [&](uint32_t m) { return msgs[m].end; });
        cudaStream_t s = e->stream;
        const tfplan::Plan& pl = pd->plan; const size_t nc = pl.in_schema.size();
        // ---- options (AuxParserOpts, generic_parser.go:41-84)
        bool add_rest = false, add_dedupe = false, nka = false, use_numbers = false, b64 = false; std::string partition;
        if (opts_json && *opts_json) {
            auto v = tfj::parse(opts_json);
            add_rest = v->get_bool("add_rest"); add_dedupe = v->get_bool("add_dedupe_keys"); nka = v->get_bool("null_keys_allowed");
            use_numbers = v->get_bool("use_numbers_in_any"); b64 = v->get_bool("unpack_bytes_base64"); partition = v->get_str("partition");
            for (const char* k : {"unescape_string_values", "add_system_columns", "add_topic_column", "infer_time_zone", "ignore_column_paths", "mask_secrets"})
                if (v->get_bool(k)) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, std::string("json parser option not handled on the device: ") + k);
            for (const char* k : {"time_field", "table_splitter"}) if (v->get(k) && v->get(k)->kind != tfj::Value::Null) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, std::string("json parser option not handled on the device: ") + k);
        }
        const size_t naux = (add_rest ? 1 : 0) + (add_dedupe ? 4 : 0);
        if (nc < naux || nc > JSN_MAX_COLS) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "json parser: the result schema must hold the aux columns and at most 128 columns");
        const size_t nf = nc - naux;
        // ---- columns
        std::vector<JsnColDev> hc(nc); std::vector<uint8_t> names; int nslots = 0;
        for (size_t c = 0; c < nc; c++) {
            const tfplan::ColSchema& cs = pl.in_schema[c]; JsnColDev& d = hc[c]; std::memset(&d, 0, sizeof d);
            d.tf = cs.tf; d.w = in_width(cs.tf); d.slot = d.w ? -1 : nslots++; d.key = cs.key; d.required = cs.required || cs.key;      // newColSchema: a key is required (:102-113)
            d.name_off = (uint32_t)names.size(); d.name_len = (uint32_t)cs.name.size(); names.insert(names.end(), cs.name.begin(), cs.name.end());
            if (c < nf) {
                switch (cs.tf) { case TF_INT8: case TF_INT16: case TF_INT32: case TF_INT64: case TF_UINT8: case TF_UINT16: case TF_UINT32: case TF_UINT64:
                                 case TF_DOUBLE: case TF_BOOLEAN: case TF_UTF8: case TF_BYTES: case TF_ANY: case TF_DATETIME: break;
                                 default: throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "json parser: field '" + cs.name + "' has a type the device parser does not handle (" + cs.type + ")"); }
                if (!cs.path.empty()) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "json parser: nested column paths are not handled on the device");
                for (size_t k = 0; k < c; k++) if (pl.in_schema[k].name == cs.name) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "json parser: duplicate column name " + cs.name);
            }
        }
        {   // addAuxFields order and types (:115-164)
            size_t c = nf; bool ok = true;
            if (add_rest) ok = ok && pl.in_schema[c++].tf == TF_ANY;
            if (add_dedupe) ok = ok && pl.in_schema[c].tf == TF_TIMESTAMP && pl.in_schema[c + 1].tf == TF_BYTES && pl.in_schema[c + 2].tf == TF_UINT64 && pl.in_schema[c + 3].tf == TF_UINT32;
            if (!ok) throw tfplan::FatalError(TF_E_FATAL_CONFIG, "json parser: the plan schema does not end with the aux columns the options add (_rest any; _timestamp timestamp, _partition string, _offset uint64, _idx uint32)");
        }
        const uint32_t part_off = (uint32_t)names.size(); names.insert(names.end(), partition.begin(), partition.end());
        // ---- text and message table into HBM
        const uint8_t* d_text = bytes;
        if (mem == TF_MEM_HOST) { e->csv_text.ensure(len + 64); if (len) CK(cudaMemcpyAsync(e->csv_text.p, bytes, len, cudaMemcpyHostToDevice, s)); d_text = e->csv_text.p; }
        const uint32_t nblk = (uint32_t)((len + CSV_NL_BLOCK - 1) / CSV_NL_BLOCK);
        const size_t bits_words = (size_t)(len / 32 + 2);
        std::vector<uint64_t> h_end(n_msgs ? n_msgs : 1), h_off(n_msgs ? n_msgs : 1); std::vector<int64_t> h_ws(n_msgs ? n_msgs : 1); std::vector<uint32_t> h_wn(n_msgs ? n_msgs : 1);
        for (uint32_t m = 0; m < n_msgs; m++) { h_end[m] = msgs[m].end; h_off[m] = msgs[m].offset; h_ws[m] = msgs[m].write_sec; h_wn[m] = msgs[m].write_nsec; }
        {
            ArenaLayout need;
            const size_t w_cnt = need(((size_t)nblk + 64) * 4), w_off = need(((size_t)nblk + 64) * 4), w_bits = need(bits_words * 4),
                         w_end = need((size_t)n_msgs * 8), w_moff = need((size_t)n_msgs * 8), w_ws = need((size_t)n_msgs * 8), w_wn = need((size_t)n_msgs * 4), w_r0 = need((size_t)n_msgs * 4);
            e->json_msgs.ensure(need.total + 256);                // message table + line-count scratch live here until the text heap is sized
            uint8_t* W = e->json_msgs.p;
            uint32_t* blk_cnt = (uint32_t*)(W + w_cnt); uint32_t* blk_off = (uint32_t*)(W + w_off); uint32_t* endbits = (uint32_t*)(W + w_bits);
            uint64_t nlines = 0;
            e->prof_n = 0;
            if (nblk) {
                CK(cudaMemsetAsync(e->d_state, 0, sizeof(DState), s));
                CK(cudaMemsetAsync(endbits, 0, bits_words * 4, s));
                CK(cudaMemcpyAsync(W + w_end, h_end.data(), (size_t)n_msgs * 8, cudaMemcpyHostToDevice, s)); CK(cudaMemcpyAsync(W + w_moff, h_off.data(), (size_t)n_msgs * 8, cudaMemcpyHostToDevice, s));
                CK(cudaMemcpyAsync(W + w_ws, h_ws.data(), (size_t)n_msgs * 8, cudaMemcpyHostToDevice, s)); CK(cudaMemcpyAsync(W + w_wn, h_wn.data(), (size_t)n_msgs * 4, cudaMemcpyHostToDevice, s));
                e->prof_begin("k_json_mark_msgs", s); launch_k_json_mark_msgs((n_msgs + 255) / 256, 256, 0, s, (const uint64_t*)(W + w_end), n_msgs, endbits); e->prof_end(s);
                e->prof_begin("k_csv_count_nl", s); launch_k_csv_count_nl(nblk, 256, 0, s, d_text, len, blk_cnt, endbits); e->prof_end(s);
                e->prof_begin("k_scan_blockcnt", s); launch_k_scan_blockcnt(1, 1024, 0, s, blk_cnt, blk_off, nblk, e->d_state); e->prof_end(s);
                DState st; CK(cudaMemcpyAsync(&st, e->d_state, sizeof st, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
                nlines = st.n_kept;
            }
            const uint64_t nrows = nlines;
            // ---- staging layout (csv_stage arena)
            ArenaLayout sneed;
            const uint32_t nlb = (uint32_t)((nlines + 127) / 128);
            const size_t o_line = sneed((nlines + 1) * 4), o_rank = sneed((nlines + 2) * 4), o_lcnt = sneed(((size_t)nlb + 64) * 4), o_loff = sneed(((size_t)nlb + 64) * 4),
                         o_err = sneed(nrows), o_ecol = sneed(nrows), o_cols = sneed(nc * sizeof(JsnColDev)), o_names = sneed(names.size()),
                         o_ss = sneed((size_t)nf * nrows * 4), o_sl = sneed((size_t)nf * nrows * 4), o_len = sneed((size_t)nslots * nrows * 4),
                         o_off = sneed((size_t)nslots * (nrows + 1) * 4), o_tot = sneed((size_t)nslots * 8 + 8), o_base = sneed((size_t)nslots * 8 + 8);
            std::vector<size_t> o_val(nc), o_aux(nc), o_vld(nc);
            for (size_t c = 0; c < nc; c++) {
                o_val[c] = hc[c].w ? sneed((size_t)hc[c].w * nrows) : 0;
                const int tf = hc[c].tf;
                o_aux[c] = (tf == TF_DATE || tf == TF_DATETIME || tf == TF_TIMESTAMP) ? sneed(4 * nrows) : (tf == TF_ANY ? sneed(nrows) : 0);
                o_vld[c] = sneed((nrows / 32 + 2) * 4);
            }
            e->csv_stage.ensure(sneed.total + 256);
            uint8_t* B = e->csv_stage.p;
            for (size_t c = 0; c < nc; c++) {
                if (hc[c].w) hc[c].values = B + o_val[c];
                const int tf = hc[c].tf;
                if (tf == TF_DATE || tf == TF_DATETIME || tf == TF_TIMESTAMP) hc[c].aux32 = (uint32_t*)(B + o_aux[c]);
                if (tf == TF_ANY) hc[c].aux8 = B + o_aux[c];
                hc[c].validity = (uint32_t*)(B + o_vld[c]);
            }
            VarHeaps heaps(nslots);
            uint32_t n_nonempty = 0;
            if (nrows) {
                CK(cudaMemcpyAsync(B + o_cols, hc.data(), nc * sizeof(JsnColDev), cudaMemcpyHostToDevice, s));
                CK(cudaMemcpyAsync(B + o_names, names.data(), names.size(), cudaMemcpyHostToDevice, s));
                CK(cudaMemsetAsync(B + o_sl, 0, (size_t)nf * nrows * 4, s));
                e->prof_begin("k_csv_line_index", s); launch_k_csv_line_index(nblk, 256, 0, s, d_text, len, blk_off, (uint32_t*)(B + o_line), endbits); e->prof_end(s);
                e->prof_begin("k_json_count_nonempty", s); launch_k_json_count_nonempty(nlb, 128, 0, s, d_text, (const uint32_t*)(B + o_line), nlines, (uint32_t*)(B + o_lcnt)); e->prof_end(s);
                e->prof_begin("k_scan_blockcnt", s); launch_k_scan_blockcnt(1, 1024, 0, s, (const uint32_t*)(B + o_lcnt), (uint32_t*)(B + o_loff), nlb, e->d_state); e->prof_end(s);
                e->prof_begin("k_json_rank", s); launch_k_json_rank(nlb, 128, 0, s, d_text, (const uint32_t*)(B + o_line), nlines, (const uint32_t*)(B + o_loff), (uint32_t*)(B + o_rank)); e->prof_end(s);
                e->prof_begin("k_json_msg_first", s); launch_k_json_msg_first((n_msgs + 255) / 256, 256, 0, s, (const uint64_t*)(W + w_end), n_msgs, (const uint32_t*)(B + o_line), nlines, (const uint32_t*)(B + o_rank), (uint32_t*)(W + w_r0)); e->prof_end(s);
                JsnArgs ja; std::memset(&ja, 0, sizeof ja);
                ja.text = d_text; ja.len = len; ja.line_end = (const uint32_t*)(B + o_line); ja.nlines = nlines;
                ja.msg_end = (const uint64_t*)(W + w_end); ja.msg_offset = (const uint64_t*)(W + w_moff); ja.msg_wsec = (const int64_t*)(W + w_ws); ja.msg_wnsec = (const uint32_t*)(W + w_wn); ja.nmsgs = n_msgs;
                ja.rank = (const uint32_t*)(B + o_rank); ja.msg_rank0 = (const uint32_t*)(W + w_r0);
                ja.cols = (const JsnColDev*)(B + o_cols); ja.ncols = (int)nc; ja.nfields = (int)nf; ja.names = B + o_names;
                ja.add_rest = add_rest; ja.add_dedupe = add_dedupe; ja.null_keys_allowed = nka; ja.use_numbers = use_numbers; ja.unpack_b64 = b64;
                ja.part_off = part_off; ja.part_len = (uint32_t)partition.size();
                ja.span_start = (uint32_t*)(B + o_ss); ja.span_len = (uint32_t*)(B + o_sl); ja.out_len = (uint32_t*)(B + o_len);
                ja.err = B + o_err; ja.errcol = B + o_ecol;
                e->prof_begin("k_json_pass1", s); launch_k_json_pass1(nlb, 128, JSN_STAGE, s, ja); e->prof_end(s);
                CK(cudaMemcpyAsync(&n_nonempty, (uint32_t*)(B + o_rank) + nlines, 4, cudaMemcpyDeviceToHost, s));
                if (nslots) {
                    place_heaps(e, heaps, (const uint32_t*)(B + o_len), nrows, nslots, (uint32_t*)(B + o_off), (uint64_t*)(B + o_tot), (uint64_t*)(B + o_base), "json batch");
                    JsnWriteArgs wa{ja, (const uint32_t*)(B + o_off), heaps.heap, (const uint64_t*)(B + o_base)};
                    e->prof_begin("k_json_pass2", s); launch_k_json_pass2(nlb, 128, JSN_STAGE, s, wa); e->prof_end(s);
                } else CK(cudaStreamSynchronize(s));
            }
            std::vector<tf_col> dev;
            auto r = chain_parsed(e, *pd, parsed_batch(hc, nrows, (const uint32_t*)(B + o_off), heaps, dev), nullptr, nrows ? B + o_err : nullptr, wire_fmt);
            // row errors: row = index among the NON-EMPTY lines (empty lines are not lines to the reference, :528-530), term = column
            if (!r->errs.empty()) {
                std::vector<uint8_t> ecol(nrows); CK(cudaMemcpyAsync(ecol.data(), B + o_ecol, nrows, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s));
                std::vector<tf_rowerr> keep; uint32_t empties = 0;
                for (auto& x : r->errs) { if (x.code == JSN_EMPTY) { empties++; continue; } tf_rowerr y = x; if (y.term == 0xff) y.term = ecol[x.row]; y.row = x.row - empties; keep.push_back(y); }
                r->errs.swap(keep);
            }
            r->rows_in = n_nonempty;
            r->consumed = len;
            *out = r.release();
        }
        return TF_OK;
    });
}

// ---------------------------------------------------------------------------------------------- Debezium
// parsers.Parser.DoBatch of the Debezium parser (pkg/parsers/registry/debezium/engine/parser.go:34-137 over
// pkg/debezium/receiver.go:142-220) fused with the transformer chain and the sink encode.
namespace {
struct DbzHostField { std::string name; int recv, scale, tf; bool key; };
// receiveTableSchema / receiveFieldColSchema (receiver.go:46-62, receiver_engine.go:104-141) with the default receivers
std::vector<DbzHostField> dbz_fields(const tfj::Value& schema, const char* which) {
    const tfj::Value* fields = schema.get("fields"); const tfj::Value* node = nullptr;
    if (fields && fields->kind == tfj::Value::Arr) for (auto& f : fields->arr) if (f->get_str("field") == which) node = f.get();
    if (!node) throw tfplan::FatalError(TF_E_FATAL_CONFIG, std::string("debezium schema has no '") + which + "' struct");
    std::vector<DbzHostField> out; const tfj::Value* fs = node->get("fields");
    if (fs && fs->kind == tfj::Value::Arr) for (auto& f : fs->arr) {
        DbzHostField h; h.name = f->get_str("field"); h.scale = 0; h.key = !f->get_bool("optional");
        const std::string kt = f->get_str("type"), nm = f->get_str("name");
        if (const tfj::Value* oti = f->get("__dt_original_type_info")) if (oti->kind == tfj::Value::Obj && !oti->get_str("original_type").empty())
            throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "debezium: database specific receivers (original types) are not handled on the device");
        if (kt == "int8") { h.recv = DR_INT8; h.tf = TF_INT8; } else if (kt == "int16") { h.recv = DR_INT16; h.tf = TF_INT16; } else if (kt == "int32") { h.recv = DR_INT32; h.tf = TF_INT32; }
        else if (kt == "int64") { h.recv = DR_INT64; h.tf = TF_INT64; } else if (kt == "boolean") { h.recv = DR_BOOL; h.tf = TF_BOOLEAN; } else if (kt == "string") { h.recv = DR_STRING; h.tf = TF_UTF8; }
        else if (kt == "float" || kt == "double") { h.recv = DR_F64; h.tf = TF_DOUBLE; }
        else if (kt == "bytes") {
            if (nm == "org.apache.kafka.connect.data.Decimal") { h.recv = DR_DECIMAL; h.tf = TF_UTF8; const tfj::Value* pa = f->get("parameters"); const std::string sc = pa ? pa->get_str("scale") : ""; if (!sc.empty()) h.scale = atoi(sc.c_str()); }
            else { h.recv = DR_BYTES; h.tf = TF_BYTES; }
        } else if (kt == "struct" && nm == "io.debezium.data.geometry.Point") { h.recv = DR_POINT; h.tf = TF_UTF8; }
        else if (kt == "struct" && nm == "io.debezium.data.VariableScaleDecimal") { h.recv = DR_VSD; h.tf = TF_DOUBLE; }
        else throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "debezium: field '" + h.name + "' of kafka type " + kt + " / " + nm + " has no default receiver on the device");
        out.push_back(h);
    }
    return out;
}
// The table fields of an envelope schema: those of its `after` struct, which the `before` struct must repeat.
std::vector<DbzHostField> dbz_table_fields(const tfj::Value& schema) {
    const std::vector<DbzHostField> fs = dbz_fields(schema, "after"), fb = dbz_fields(schema, "before");
    auto same = [](const DbzHostField& a, const DbzHostField& b) { return a.name == b.name && a.recv == b.recv && a.scale == b.scale; };
    if (!std::equal(fs.begin(), fs.end(), fb.begin(), fb.end(), same)) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "debezium: 'before' and 'after' structs differ");
    return fs;
}
}  // namespace

// Host-only: the table schema and receivers tfgpu_parse_debezium derives from a Kafka Connect envelope schema (no GPU needed):
// [{"name","type","key","recv","scale"}, ...] in the order of the `after` struct, or the error the call would return.
int tfgpu_debezium_schema_validate(const char* schema_text, char* describe_out, uint64_t cap, char* err_out, uint64_t err_cap) {
    if (!schema_text) return TF_E_FATAL_ARG;
    return validated(describe_out, cap, err_out, err_cap, [&] {
        const std::vector<DbzHostField> fs = dbz_table_fields(*tfj::parse(schema_text));
        static const char* yt[] = {"", "int8", "int16", "int32", "int64", "uint8", "uint16", "uint32", "uint64", "float", "double", "boolean", "string", "utf8", "any", "date", "datetime", "timestamp", "interval"};
        std::string d = "[";
        for (size_t i = 0; i < fs.size(); i++) {
            if (i) d += ",";
            d += "{\"name\":" + host_json_quote_nohtml(fs[i].name) + ",\"type\":\"" + yt[fs[i].tf] + "\",\"key\":" + (fs[i].key ? "true" : "false") +
                 ",\"recv\":" + std::to_string(fs[i].recv) + ",\"scale\":" + std::to_string(fs[i].scale) + "}";
        }
        return d + "]";
    });
}

int tfgpu_parse_debezium(tfgpu_engine* e, int plan_id, const char* opts_json, const uint8_t* bytes, uint64_t len, int mem,
                         const uint64_t* msg_ends, uint32_t n_msgs, int wire_fmt, tfgpu_result** out) {
    PlanDev* pd = plan_arg(e, plan_id);
    if (!pd || !out || !opts_json || (!bytes && len) || (!msg_ends && n_msgs)) return TF_E_FATAL_ARG;
    *out = nullptr;
    return guarded(e, [&] {
        if (len >= (1ull << 32) - 16) throw tfplan::FatalError(TF_E_FATAL_ARG, "debezium batch must be < 4 GiB");
        check_wire(*pd, wire_fmt, true);
        check_msg_ends(len, n_msgs, [&](uint32_t m) { return msg_ends[m]; });
        cudaStream_t s = e->stream;
        const tfplan::Plan& pl = pd->plan; const size_t nc = pl.in_schema.size();
        auto ov = tfj::parse(opts_json);
        const std::string schema_text = ov->get_str("schema_text");
        const bool use_sr = ov->get_bool("schema_registry"), check_table = ov->get_bool("check_table");
        const uint32_t schema_id = (uint32_t)ov->get_num("schema_id", 0);
        if (schema_text.empty()) throw tfplan::FatalError(TF_E_FATAL_CONFIG, "debezium: opts.schema_text (the Kafka Connect schema this plan was built for) is required");
        const std::vector<DbzHostField> fs = dbz_table_fields(*tfj::parse(schema_text.c_str()));
        if (fs.size() != nc || nc > JSN_MAX_COLS) throw tfplan::FatalError(TF_E_FATAL_CONFIG, "debezium: the plan schema must be the table schema of the 'after' struct (at most 128 columns)");
        std::vector<DbzColDev> hc(nc); std::vector<uint8_t> names; int nslots = 0;
        for (size_t c = 0; c < nc; c++) {
            const tfplan::ColSchema& cs = pl.in_schema[c]; DbzColDev& d = hc[c]; std::memset(&d, 0, sizeof d);
            if (cs.name != fs[c].name || cs.tf != fs[c].tf) throw tfplan::FatalError(TF_E_FATAL_CONFIG, "debezium: plan column '" + cs.name + "' does not match the schema field '" + fs[c].name + "' (receiveFieldColSchema type)");
            for (size_t k = 0; k < c; k++) if (fs[k].name == fs[c].name) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "debezium: duplicate field " + fs[c].name);
            for (unsigned char ch : fs[c].name) if (ch >= 0x80 || ch == '\\' || ch == '"' || ch < 0x20) throw tfplan::FatalError(TF_E_FATAL_UNSUPPORTED, "debezium: field names must be plain ASCII on the device");
            d.recv = fs[c].recv; d.scale = fs[c].scale; d.tf = cs.tf; d.w = in_width(cs.tf); d.slot = d.w ? -1 : nslots++; d.key = fs[c].key;
            d.name_off = (uint32_t)names.size(); d.name_len = (uint32_t)cs.name.size(); names.insert(names.end(), cs.name.begin(), cs.name.end());
        }
        const uint32_t ts_off = (uint32_t)names.size(); names.insert(names.end(), pl.ns.begin(), pl.ns.end());
        const uint32_t tn_off = (uint32_t)names.size(); names.insert(names.end(), pl.name.begin(), pl.name.end());
        const uint32_t st_off = (uint32_t)names.size(); names.insert(names.end(), schema_text.begin(), schema_text.end());
        const uint8_t* d_text = bytes;
        if (mem == TF_MEM_HOST) { e->csv_text.ensure(len + 64); if (len) CK(cudaMemcpyAsync(e->csv_text.p, bytes, len, cudaMemcpyHostToDevice, s)); d_text = e->csv_text.p; }
        const uint64_t n = n_msgs;
        ArenaLayout need;
        const size_t o_end = need(n * 8), o_err = need(n), o_ecol = need(n), o_cols = need(nc * sizeof(DbzColDev)), o_names = need(names.size()),
                     o_ss = need(nc * n * 4), o_sl = need(nc * n * 4), o_len = need((size_t)nslots * n * 4), o_off = need((size_t)nslots * (n + 1) * 4),
                     o_tot = need((size_t)nslots * 8 + 8), o_base = need((size_t)nslots * 8 + 8), o_kind = need(n), o_tx = need(n * 4), o_lsn = need(n * 8), o_ct = need(n * 8);
        std::vector<size_t> o_val(nc), o_vld(nc);
        for (size_t c = 0; c < nc; c++) { o_val[c] = hc[c].w ? need((size_t)hc[c].w * n) : 0; o_vld[c] = need((n / 32 + 2) * 4); }
        e->csv_stage.ensure(need.total + 256);
        uint8_t* B = e->csv_stage.p;
        for (size_t c = 0; c < nc; c++) { if (hc[c].w) hc[c].values = B + o_val[c]; hc[c].validity = (uint32_t*)(B + o_vld[c]); }
        VarHeaps heaps(nslots);
        e->prof_n = 0;
        if (n) {
            CK(cudaMemcpyAsync(B + o_end, msg_ends, n * 8, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(B + o_cols, hc.data(), nc * sizeof(DbzColDev), cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(B + o_names, names.data(), names.size(), cudaMemcpyHostToDevice, s));
            CK(cudaMemsetAsync(B + o_sl, 0, nc * n * 4, s));
            DbzArgs da; std::memset(&da, 0, sizeof da);
            da.text = d_text; da.msg_end = (const uint64_t*)(B + o_end); da.nmsgs = n; da.cols = (const DbzColDev*)(B + o_cols); da.ncols = (int)nc; da.names = B + o_names;
            da.schema_text = B + o_names + st_off; da.schema_len = (uint32_t)schema_text.size(); da.schema_id = schema_id; da.use_sr = use_sr; da.check_table = check_table;
            da.tbl_schema_off = ts_off; da.tbl_schema_len = (uint32_t)pl.ns.size(); da.tbl_name_off = tn_off; da.tbl_name_len = (uint32_t)pl.name.size();
            da.span_start = (uint32_t*)(B + o_ss); da.span_len = (uint32_t*)(B + o_sl); da.out_len = (uint32_t*)(B + o_len);
            da.kinds = B + o_kind; da.tx_id = (uint32_t*)(B + o_tx); da.lsn = (uint64_t*)(B + o_lsn); da.commit_time = (uint64_t*)(B + o_ct); da.err = B + o_err; da.errcol = B + o_ecol;
            const uint32_t nb = (uint32_t)((n + 127) / 128);
            e->prof_begin("k_dbz_pass1", s); launch_k_dbz_pass1(nb, 128, DBZ_STAGE, s, da); e->prof_end(s);
            if (nslots) {
                place_heaps(e, heaps, (const uint32_t*)(B + o_len), n, nslots, (uint32_t*)(B + o_off), (uint64_t*)(B + o_tot), (uint64_t*)(B + o_base), "debezium batch");
                DbzWriteArgs wa{da, (const uint32_t*)(B + o_off), heaps.heap, (const uint64_t*)(B + o_base)};
                e->prof_begin("k_dbz_pass2", s); launch_k_dbz_pass2(nb, 128, 0, s, wa); e->prof_end(s);
            }
            CK(cudaGetLastError());
        }
        std::vector<tf_col> dev;
        auto r = chain_parsed(e, *pd, parsed_batch(hc, n, (const uint32_t*)(B + o_off), heaps, dev), n ? B + o_kind : nullptr, n ? B + o_err : nullptr, wire_fmt);
        if (n) {
            if (!r->errs.empty()) { std::vector<uint8_t> ecol(n); CK(cudaMemcpyAsync(ecol.data(), B + o_ecol, n, cudaMemcpyDeviceToHost, s)); CK(cudaStreamSynchronize(s)); for (auto& x : r->errs) if (x.term == 0xff) x.term = ecol[x.row]; }
            r->meta_kinds.resize(n); r->meta_tx.resize(n); r->meta_lsn.resize(n); r->meta_ct.resize(n); r->selection.resize(r->rows_out);
            CK(cudaMemcpyAsync(r->meta_kinds.data(), B + o_kind, n, cudaMemcpyDeviceToHost, s)); CK(cudaMemcpyAsync(r->meta_tx.data(), B + o_tx, n * 4, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(r->meta_lsn.data(), B + o_lsn, n * 8, cudaMemcpyDeviceToHost, s)); CK(cudaMemcpyAsync(r->meta_ct.data(), B + o_ct, n * 8, cudaMemcpyDeviceToHost, s));
            if (r->rows_out) CK(cudaMemcpyAsync(r->selection.data(), e->sel, r->rows_out * 4, cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
        }
        r->consumed = len;
        *out = r.release();
        return TF_OK;
    });
}

// debug / profiling aid: cycles thread 0 of every k_lz4_frames CTA spent per phase since enabling (stage, match, parse, scan, emit)
int tfgpu_debug_lz4_phases(tfgpu_engine* e, int enable, uint64_t out[8]) {
    if (!e) return TF_E_FATAL_ARG;
    return guarded(e, [&] {
        if (enable && !e->lz_phases) { CK(cudaMalloc(&e->lz_phases, 64)); CK(cudaMemset(e->lz_phases, 0, 64)); }
        if (out && e->lz_phases) { CK(cudaStreamSynchronize(e->stream)); CK(cudaMemcpy(out, e->lz_phases, 64, cudaMemcpyDeviceToHost)); CK(cudaMemset(e->lz_phases, 0, 64)); }
        if (!enable && e->lz_phases) { CK(cudaFree(e->lz_phases)); e->lz_phases = nullptr; }
        return TF_OK;
    });
}

const uint32_t* tfgpu_result_dbz_msg_sizes(const tfgpu_result* r) { return (r && !r->msg_sizes.empty()) ? r->msg_sizes.data() : nullptr; }
const uint32_t* tfgpu_result_selection(const tfgpu_result* r) { return (r && !r->selection.empty()) ? r->selection.data() : nullptr; }
const uint8_t* tfgpu_result_meta_kinds(const tfgpu_result* r) { return (r && !r->meta_kinds.empty()) ? r->meta_kinds.data() : nullptr; }
const uint32_t* tfgpu_result_meta_tx_id(const tfgpu_result* r) { return (r && !r->meta_tx.empty()) ? r->meta_tx.data() : nullptr; }
const uint64_t* tfgpu_result_meta_lsn(const tfgpu_result* r) { return (r && !r->meta_lsn.empty()) ? r->meta_lsn.data() : nullptr; }
const uint64_t* tfgpu_result_meta_commit_time(const tfgpu_result* r) { return (r && !r->meta_ct.empty()) ? r->meta_ct.data() : nullptr; }

uint64_t tfgpu_result_consumed(const tfgpu_result* r) { return r ? r->consumed : 0; }

uint64_t tfgpu_result_rows_in(const tfgpu_result* r) { return r ? r->rows_in : 0; }
uint64_t tfgpu_result_rows_out(const tfgpu_result* r) { return r ? r->rows_out : 0; }
uint64_t tfgpu_result_n_errors(const tfgpu_result* r) { return r ? r->errs.size() : 0; }
const tf_rowerr* tfgpu_result_errors(const tfgpu_result* r) { return (r && !r->errs.empty()) ? r->errs.data() : nullptr; }
const tf_batch* tfgpu_result_batch(const tfgpu_result* r) { return (r && r->batch.ncols) ? &r->batch : nullptr; }
const uint8_t* tfgpu_result_bytes(const tfgpu_result* r) { return r ? r->bytes : nullptr; }
uint64_t tfgpu_result_bytes_len(const tfgpu_result* r) { return r ? r->bytes_len : 0; }
uint64_t tfgpu_result_raw_len(const tfgpu_result* r) { return r ? r->raw_len : 0; }
uint64_t tfgpu_result_n_frames(const tfgpu_result* r) { return r ? r->n_frames : 0; }
const uint32_t* tfgpu_result_part_ids(const tfgpu_result* r) { return (r && !r->part_ids.empty()) ? r->part_ids.data() : nullptr; }
const uint32_t* tfgpu_result_key_sizes(const tfgpu_result* r) { return (r && !r->key_sizes.empty()) ? r->key_sizes.data() : nullptr; }
const uint32_t* tfgpu_result_row_sizes(const tfgpu_result* r) { return (r && !r->row_sizes.empty()) ? r->row_sizes.data() : nullptr; }

// queue JSON serializer batching (pkg/serializer/queue/json_batcher.go:13-66): host only, no device needed
int tfgpu_queue_debezium_batches(const uint32_t* value_sizes, uint64_t n, uint64_t max_message_size, uint64_t* starts, uint64_t cap, uint64_t* n_msgs) {
    if ((!value_sizes && n) || !starts || !n_msgs) return TF_E_FATAL_ARG;
    uint64_t k = 0, cur = 0;
    for (uint64_t i = 0; i < n; i++) {
        // expandArrIfNeeded :76-86: a new message for the first value and whenever len(last) + 1 + len(new) > maxMessageSize;
        // without a limit every value stays its own message (MergeBack :53-65)
        if (i == 0 || !max_message_size || cur + 1 + value_sizes[i] > max_message_size) { if (k >= cap) return TF_E_FATAL_ARG; starts[k++] = i; cur = 0; }
        cur += value_sizes[i];
    }
    if (k >= cap) return TF_E_FATAL_ARG;
    starts[k] = n; *n_msgs = k;
    return TF_OK;
}
int tfgpu_queue_json_batches(const uint32_t* row_sizes, uint64_t n, uint64_t max_message_size, uint64_t max_change_items, uint64_t* starts, uint64_t cap, uint64_t* n_msgs) {
    if ((!row_sizes && n) || !starts || !n_msgs) return TF_E_FATAL_ARG;
    uint64_t k = 0, start = 0, sum = 0;
    auto emit = [&](uint64_t s) -> bool { if (k >= cap) return false; starts[k++] = s; return true; };
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t count = i - start + 1;
        const bool viol = (max_message_size && sum + (count - 1) + row_sizes[i] > max_message_size) || (max_change_items && count > max_change_items);
        if (!viol) { sum += row_sizes[i]; continue; }
        if (!emit(start)) return TF_E_FATAL_ARG;
        if (i == start) { start = i + 1; sum = 0; }        // a single item over the size limit goes out alone
        else { start = i; sum = row_sizes[i]; }
    }
    if (start != n && !emit(start)) return TF_E_FATAL_ARG;
    if (k >= cap) return TF_E_FATAL_ARG;
    starts[k] = n; *n_msgs = k;
    return TF_OK;
}
void tfgpu_result_release(tfgpu_result* r) {
    if (!r) return;
    if (r->bytes && r->bytes_pinned) cudaFreeHost(r->bytes);   // otherwise the engine's landing buffer
    for (auto p : r->owned) free(p);
    delete r;
}

}  // extern "C"
