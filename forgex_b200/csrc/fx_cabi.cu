// fx_cabi.cu -- the C ABI of include/forgex_b200.h: pattern handles, table upload, kernel launches.
// Product code; never links oracle/.  No CPU fallback: every matching entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/forgex_b200.h"
#include "fx_internal.hpp"
#include "fx_kernels.cuh"

using namespace fxk;

namespace {

std::atomic<long long> g_launches{0};

constexpr int STATE_CAP = 16383;                 // Forgex's own ceiling (lazy_dfa_graph_m.F90:90-92 with parameters_m.f90:126-130)
constexpr int SPARSE_STATE_CAP = 2048;           // optional anchored automaton of a prefix-less `.in.` pattern
constexpr int DIRECT_LIMIT_BYTES = 40 * 1024;    // 256-column table kept in shared memory up to this size
constexpr int SMEM_TABLE_LIMIT_BYTES = 160 * 1024;
constexpr int SPAN_DIRECT_MAX_STATES = 127;      // span forward table as padded 256-column rows in shared memory (<= 64 KB)
constexpr int SPAN_CLASSED_SMEM_BYTES = 96 * 1024;
constexpr int SPAN_REV_SMEM_BYTES = 24 * 1024;

struct DeviceTables {
    int device = -1;
    uint16_t* table = nullptr;   // class-compressed
    uint16_t* direct = nullptr;  // 256 columns (only when small)
    uint8_t* table8 = nullptr;   // 256 columns, one byte per entry (boolean tables with <= 255 states)
    uint8_t* classmap = nullptr;
    uint8_t* flags = nullptr;
    uint8_t* lits = nullptr;
    // anchored (REGEX-mode) tables of an `.in.` pattern with an active prefix
    uint16_t* a_table = nullptr;
    uint8_t* a_classmap = nullptr;
    uint8_t* a_flags = nullptr;
    // linear-time span path (FX_OP_REGEX, when the pattern has one)
    uint16_t* sp_table = nullptr; uint16_t* sp_direct = nullptr;
    uint8_t* sp_classmap = nullptr; uint8_t* sp_endinfo = nullptr;
    uint16_t* r_delta = nullptr; int32_t* r_cuts = nullptr; uint8_t* r_page = nullptr; uint8_t* r_mixed = nullptr;
    uint16_t* sm_reach = nullptr; uint16_t* sm_img = nullptr; uint8_t* sm_sync = nullptr;
    uint16_t* ctab4 = nullptr; uint8_t* cmap4 = nullptr;       // compact ASCII-columns table of a big boolean automaton (K1c)
    uint64_t* nfa_trans = nullptr; uint64_t* nfa_q0 = nullptr; int32_t* nfa_cuts = nullptr;     // NFA engine (patterns past the state cap)
    uint8_t* w_work = nullptr; size_t w_work_cap = 0;
    // grow-only scratch for the host-pointer entry points
    uint8_t* w_buf = nullptr; size_t w_buf_cap = 0;
    int64_t* w_off = nullptr; size_t w_off_cap = 0;
    uint8_t* w_out = nullptr; size_t w_out_cap = 0;
    int64_t* w_span = nullptr; size_t w_span_cap = 0;
    unsigned long long* w_best = nullptr;
    int sm_count = 0;
};

// first-byte set F of an anchored automaton: at most 4 ASCII ranges, plus "some bytes >= 0xC0"
struct FirstSet {
    int nr = 0;
    uint8_t lo[4] = {0, 0, 0, 0}, hi[4] = {0, 0, 0, 0};
    bool high = false;
    int sweep_nr = 0;            // the ranges the sweep tests: lo/hi with close neighbours merged (a superset of F)
    uint8_t sweep_lo[4] = {0, 0, 0, 0}, sweep_hi[4] = {0, 0, 0, 0};
    bool two = false;            // one first byte, and after it one ASCII byte (plus, maybe, lead bytes) keeps the automaton alive
    uint8_t second = 0;
    bool second_high = false;
};

}  // namespace

struct fx_pattern {
    fx::Program prog;
    int residency = FX_TABLE_AUTO;
    int last_residency = 0, last_direct = 0;
    fx::Program anchored;        // FX_OP_IN: the anchored (REGEX-mode) automaton, for the prefix replay and for K2c
    bool has_anchored = false;
    int prefix_mode = 0;         // see KParams::prefix_mode
    bool prefix_scan = false;    // FX_OP_REGEX: the long-buffer path can take the prefix literal's occurrences as its candidates
    bool prefix_neutral = false; // ... and every match provably begins with the literal (prefilter_is_neutral)
    // long-buffer state-map scan (K5): reachable live states of the span forward automaton and, per byte value, the
    // image of ALL of them under that byte (count, then up to SM_M states; 0xFFFF = wider)
    std::vector<uint16_t> sm_reach, sm_img;
    uint8_t sm_sync[256];        // synchronising bytes (see StateMapParams::sync)
    bool statemap = false;
    int last_statemap = 0;       // 1: the last fx_regex_buffer* call was answered by the state-map scan
    // K1c: the ASCII columns of a big boolean table (at most 4 byte classes among the ASCII bytes): nstates x 4 words
    std::vector<uint16_t> ctab4;
    uint8_t cmap4[256];
    bool compact = false;
    int last_compact = 0;
    FirstSet first;              // bytes that survive the first step out of q0 of the anchored automaton
    bool sparse = false;         // the sparse-start kernel (K2c) may serve `.in.` batches
    int last_sparse = 0;
    DeviceTables dev;
    std::mutex mu;               // serialises the host-pointer entry points (they share the grow-only scratch)
    std::mutex dev_mu;           // serialises the lazy upload of the tables (ensure_device)
    bool dev_touched = false;    // some allocation may exist even if the upload failed half-way
};

namespace {

#define CUDA_TRY(expr)                                        \
    do {                                                      \
        cudaError_t e__ = (expr);                             \
        if (e__ != cudaSuccess) return cuda_status(e__);      \
    } while (0)

int cuda_status(cudaError_t e) {
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInitializationError) return FX_ERR_NO_DEVICE;
    return -(int)e;
}

// Is Forgex's prefix prefilter (api_internal_m.F90:76-104, utility_m.f90:58-117) result-neutral for
// this pattern as long as the text is pure ASCII, so that trying every character boundary gives the
// same answer?  Sufficient: the suffix is blank; the prefix has no border (occurrences cannot overlap,
// so the non-overlapping occurrence list is the full list), holds no NUL, and is a true prefix of every
// match: walking its code points from q0 in the anchored automaton, every other class is dead and no
// accept is seen before it ends.  (With bytes >= 0x80 in the text an overlong encoding could start a
// match that the byte-wise prefix search does not see; the kernels re-check such texts exactly.)
bool prefilter_is_neutral(const fx::Program& anchored) {
    const std::string& pre = anchored.lit.prefix;
    if (fx::fortran_blank(pre)) return true;
    if (!fx::fortran_blank(anchored.lit.suffix)) return false;
    if (pre.find('\0') != std::string::npos) return false;
    size_t n = pre.size();
    for (size_t k = 1; k < n; k++)
        if (pre.compare(0, k, pre, n - k, k) == 0) return false;   // border
    for (unsigned char c : pre) if (c >= 0x80) return false;         // keep the argument to ASCII prefixes
    const fx::CpAutomaton& a = anchored.cp;
    int st = a.q0;
    for (size_t i = 0; i < n; i++) {
        if (i > 0 && a.accept[(size_t)st]) return false;
        int want = a.class_of((unsigned char)pre[i]);
        if (a.cuts[(size_t)want] != (unsigned char)pre[i] || a.cuts[(size_t)want + 1] != (unsigned char)pre[i] + 1) return false;
        for (int c = 0; c < a.nclasses; c++)
            if (c != want && a.delta[(size_t)st * (size_t)a.nclasses + (size_t)c] != 0) return false;
        st = a.delta[(size_t)st * (size_t)a.nclasses + (size_t)want];
        if (st == 0) return false;
    }
    return true;
}

// route overrides (environment, read per call): tests and tools force a kernel or a path that the default choice
// would not take for their input, to check it against the oracle.  DESIGN.md lists them.
int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// Can the sparse-start kernel (fx_kernels.cuh, K2c) serve this `.in.` pattern?  F = bytes b with a live (or accepting)
// transition out of q0.  Required: F is non-empty, holds no continuation byte (so every candidate is a character
// boundary), its ASCII part fits 4 ranges; and the leading-NUL start does not accept by itself (no "empty winner" that would stop the
// reference's search early, api_internal_m.F90:139-150).  Worth it only when candidates are rare: without knowing the
// text, "F holds at most FX_SPARSE_MAX_FIRST (default 6) ASCII bytes" stands in for that.
bool sparse_first_set(const fx::ByteTable& at, FirstSet& fs, bool for_in) {
    fs = FirstSet();
    if (at.q0 == 0) return false;
    if (for_in && at.start_nul != 0 && (at.flags[(size_t)at.start_nul] & fxk::SF_ACC)) return false;
    bool in_f[256];
    for (int b = 0; b < 256; b++) {
        const uint16_t w = at.table[((size_t)at.q0 << at.row_shift) + at.classmap[b]];
        in_f[b] = (w & (fxk::W_STATE | fxk::W_ACC)) != 0;
    }
    for (int b = 0x80; b < 0xC0; b++) if (in_f[b]) return false;
    for (int b = 0xC0; b < 256; b++) fs.high |= in_f[b];
    int ascii = 0;
    for (int b = 0; b < 128; b++) ascii += in_f[b];
    if (ascii > env_int("FX_SPARSE_MAX_FIRST", 6)) return false;
    int b = 0;
    while (b < 128) {
        if (!in_f[b]) { b++; continue; }
        int e = b;
        while (e + 1 < 128 && in_f[e + 1]) e++;
        if (fs.nr == 4) return false;
        fs.lo[fs.nr] = (uint8_t)b; fs.hi[fs.nr] = (uint8_t)e; fs.nr++;
        b = e + 1;
    }
    if (fs.nr == 0 && !fs.high) return false;
    // Sweep ranges may over-approximate F (every candidate is confirmed by the table): neighbours at most 9 byte
    // values apart are merged -- {NUL, LF, CR}, the bytes `^` can consume, become the one range [0x00, 0x0D].
    fs.sweep_nr = 0;
    for (int r = 0; r < fs.nr; r++) {
        if (fs.sweep_nr > 0 && fs.lo[r] - fs.sweep_hi[fs.sweep_nr - 1] <= 10) fs.sweep_hi[fs.sweep_nr - 1] = fs.hi[r];
        else { fs.sweep_lo[fs.sweep_nr] = fs.lo[r]; fs.sweep_hi[fs.sweep_nr] = fs.hi[r]; fs.sweep_nr++; }
    }
    // the two-byte sweep filter: F's ASCII part is one byte V1, the step q0 -V1-> w1 neither accepts nor enters a
    // sequence, and from w1 exactly one ASCII byte V2 != NUL survives (no continuation byte does)
    if (fs.nr == 1 && fs.lo[0] == fs.hi[0]) {
        const uint16_t w1 = at.table[((size_t)at.q0 << at.row_shift) + at.classmap[fs.lo[0]]];
        if ((w1 & (fxk::W_ACC | fxk::W_INTER)) == 0 && (w1 & fxk::W_STATE) != 0) {
            int nascii = 0, v2 = 0;
            bool cont = false, hi2 = false;
            for (int c = 0; c < 256; c++) {
                const uint16_t w2 = at.table[((size_t)(w1 & fxk::W_STATE) << at.row_shift) + at.classmap[c]];
                if ((w2 & (fxk::W_STATE | fxk::W_ACC)) == 0) continue;
                if (c < 0x80) { nascii++; v2 = c; }
                else if (c < 0xC0) cont = true;
                else hi2 = true;
            }
            if (nascii == 1 && v2 != 0 && !cont) { fs.two = true; fs.second = (uint8_t)v2; fs.second_high = hi2; }
        }
    }
    return true;
}

int ensure_device(fx_pattern* p) {
    std::lock_guard<std::mutex> lock(p->dev_mu);    // two threads may make the first call on one handle
    DeviceTables& d = p->dev;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (d.device == dev) return FX_OK;
    if (d.device >= 0) return FX_ERR_BAD_ARGUMENT;  // one device per handle
    if (p->dev_touched) return FX_ERR_BAD_ARGUMENT; // an earlier upload failed half-way: the handle is unusable
    p->dev_touched = true;
    if (p->prog.nfa_engine) {                       // NFA engine: the sets, the cuts and the literals are all there is
        const fx::NfaTables& nt = p->prog.nfa_tables;
        CUDA_TRY(cudaMalloc(&d.nfa_trans, nt.trans.size() * 8 + 16));
        CUDA_TRY(cudaMemcpy(d.nfa_trans, nt.trans.data(), nt.trans.size() * 8, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.nfa_q0, nt.q0.size() * 8 + 16));
        CUDA_TRY(cudaMemcpy(d.nfa_q0, nt.q0.data(), nt.q0.size() * 8, cudaMemcpyHostToDevice));
        std::vector<int32_t> cuts(nt.cuts.begin(), nt.cuts.end());
        CUDA_TRY(cudaMalloc(&d.nfa_cuts, cuts.size() * 4 + 16));
        CUDA_TRY(cudaMemcpy(d.nfa_cuts, cuts.data(), cuts.size() * 4, cudaMemcpyHostToDevice));
        std::string lits = p->prog.lit.all + p->prog.lit.prefix + p->prog.lit.suffix;
        CUDA_TRY(cudaMalloc(&d.lits, lits.size() + 16));
        if (!lits.empty()) CUDA_TRY(cudaMemcpy(d.lits, lits.data(), lits.size(), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.w_best, 64));
        CUDA_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
        d.device = dev;
        return FX_OK;
    }
    const fx::ByteTable& bt = p->prog.bt;
    size_t tb = (bt.table.size() * 2 + 15) & ~(size_t)15, db = (bt.direct.size() * 2 + 15) & ~(size_t)15;
    CUDA_TRY(cudaMalloc(&d.table, tb + 16));
    CUDA_TRY(cudaMemset(d.table, 0, tb + 16));
    CUDA_TRY(cudaMemcpy(d.table, bt.table.data(), bt.table.size() * 2, cudaMemcpyHostToDevice));
    if ((int)db <= DIRECT_LIMIT_BYTES) {
        CUDA_TRY(cudaMalloc(&d.direct, db + 16));
        CUDA_TRY(cudaMemset(d.direct, 0, db + 16));
        CUDA_TRY(cudaMemcpy(d.direct, bt.direct.data(), bt.direct.size() * 2, cudaMemcpyHostToDevice));
    }
    if (!bt.direct8.empty()) {
        CUDA_TRY(cudaMalloc(&d.table8, bt.direct8.size() + 16));
        CUDA_TRY(cudaMemcpy(d.table8, bt.direct8.data(), bt.direct8.size(), cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMalloc(&d.classmap, 256));
    CUDA_TRY(cudaMemcpy(d.classmap, bt.classmap, 256, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&d.flags, (bt.flags.size() + 15) & ~(size_t)15));
    CUDA_TRY(cudaMemcpy(d.flags, bt.flags.data(), bt.flags.size(), cudaMemcpyHostToDevice));
    std::string lits = p->prog.lit.all + p->prog.lit.prefix + p->prog.lit.suffix;
    CUDA_TRY(cudaMalloc(&d.lits, lits.size() + 16));
    if (!lits.empty()) CUDA_TRY(cudaMemcpy(d.lits, lits.data(), lits.size(), cudaMemcpyHostToDevice));
    if (p->has_anchored) {
        const fx::ByteTable& at = p->anchored.bt;
        CUDA_TRY(cudaMalloc(&d.a_table, at.table.size() * 2 + 16));
        CUDA_TRY(cudaMemcpy(d.a_table, at.table.data(), at.table.size() * 2, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.a_classmap, 256));
        CUDA_TRY(cudaMemcpy(d.a_classmap, at.classmap, 256, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.a_flags, at.flags.size() + 16));
        CUDA_TRY(cudaMemcpy(d.a_flags, at.flags.data(), at.flags.size(), cudaMemcpyHostToDevice));
    }
    if (p->prog.has_span_tables) {
        const fx::ByteTable& st = p->prog.span_bt;
        const fx::RevAutomaton& rv = p->prog.rev;
        CUDA_TRY(cudaMalloc(&d.sp_table, st.table.size() * 2 + 32));
        CUDA_TRY(cudaMemset(d.sp_table, 0, st.table.size() * 2 + 32));
        CUDA_TRY(cudaMemcpy(d.sp_table, st.table.data(), st.table.size() * 2, cudaMemcpyHostToDevice));
        if (st.nstates <= SPAN_DIRECT_MAX_STATES) {
            CUDA_TRY(cudaMalloc(&d.sp_direct, st.direct.size() * 2 + 32));
            CUDA_TRY(cudaMemcpy(d.sp_direct, st.direct.data(), st.direct.size() * 2, cudaMemcpyHostToDevice));
        }
        CUDA_TRY(cudaMalloc(&d.sp_classmap, 256));
        CUDA_TRY(cudaMemcpy(d.sp_classmap, st.classmap, 256, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.sp_endinfo, st.endinfo.size() + 16));
        CUDA_TRY(cudaMemcpy(d.sp_endinfo, st.endinfo.data(), st.endinfo.size(), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.r_delta, rv.delta16.size() * 2 + 16));
        CUDA_TRY(cudaMemcpy(d.r_delta, rv.delta16.data(), rv.delta16.size() * 2, cudaMemcpyHostToDevice));
        std::vector<int32_t> cuts(rv.cuts.begin(), rv.cuts.end());
        CUDA_TRY(cudaMalloc(&d.r_cuts, cuts.size() * 4 + 16));
        CUDA_TRY(cudaMemcpy(d.r_cuts, cuts.data(), cuts.size() * 4, cudaMemcpyHostToDevice));
        if (!rv.page.empty()) {
            CUDA_TRY(cudaMalloc(&d.r_page, rv.page.size()));
            CUDA_TRY(cudaMemcpy(d.r_page, rv.page.data(), rv.page.size(), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMalloc(&d.r_mixed, rv.mixed.size() + 64));
            if (!rv.mixed.empty()) CUDA_TRY(cudaMemcpy(d.r_mixed, rv.mixed.data(), rv.mixed.size(), cudaMemcpyHostToDevice));
        }
    }
    if (p->compact) {
        CUDA_TRY(cudaMalloc(&d.ctab4, p->ctab4.size() * 2 + 16));
        CUDA_TRY(cudaMemcpy(d.ctab4, p->ctab4.data(), p->ctab4.size() * 2, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.cmap4, 256));
        CUDA_TRY(cudaMemcpy(d.cmap4, p->cmap4, 256, cudaMemcpyHostToDevice));
    }
    if (p->statemap) {
        CUDA_TRY(cudaMalloc(&d.sm_reach, p->sm_reach.size() * 2 + 16));
        CUDA_TRY(cudaMemcpy(d.sm_reach, p->sm_reach.data(), p->sm_reach.size() * 2, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.sm_img, p->sm_img.size() * 2 + 16));
        CUDA_TRY(cudaMemcpy(d.sm_img, p->sm_img.data(), p->sm_img.size() * 2, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&d.sm_sync, 256));
        CUDA_TRY(cudaMemcpy(d.sm_sync, p->sm_sync, 256, cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMalloc(&d.w_best, 64));
    CUDA_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
    d.device = dev;
    return FX_OK;
}

struct Plan {
    int kind;          // fxk::Table<KIND>: 0 u8 direct smem, 1 u16 direct smem, 2 classed smem, 3 classed global
    int table_bytes;   // bytes of the table staged in shared memory (0 for kind 3)
    KParams kp;
};

int make_plan(fx_pattern* p, Plan& pl) {
    const fx::ByteTable& bt = p->prog.bt;
    const DeviceTables& d = p->dev;
    const bool span = bt.flag_bits;
    int classed_bytes = (int)bt.table.size() * 2, direct_bytes = (int)bt.direct.size() * 2;
    bool direct16_ok = span && d.direct != nullptr && direct_bytes <= DIRECT_LIMIT_BYTES;
    bool direct8_ok = !span && d.table8 != nullptr;
    bool classed_smem_ok = classed_bytes <= SMEM_TABLE_LIMIT_BYTES;
    int res = p->residency;
    if (res == FX_TABLE_SMEM && !direct16_ok && !direct8_ok && !classed_smem_ok) return FX_ERR_BAD_ARGUMENT;
    if (res == FX_TABLE_GLOBAL) pl.kind = 3;
    else if (direct8_ok) pl.kind = 0;
    else if (direct16_ok) pl.kind = 1;
    else if (classed_smem_ok) pl.kind = 2;
    else pl.kind = 3;
    pl.table_bytes = pl.kind == 0 ? bt.nstates * ROW8 : pl.kind == 1 ? direct_bytes : pl.kind == 2 ? classed_bytes : 0;
    KParams& k = pl.kp;
    k.table = pl.kind == 1 ? d.direct : d.table;
    k.table8 = d.table8;
    k.ctable = d.table;
    k.classmap = d.classmap;
    k.flags = d.flags;
    k.lits = d.lits;
    k.table_words = (pl.kind == 1 ? direct_bytes : classed_bytes) / 2;
    k.nstates = bt.nstates;
    k.row_shift = pl.kind == 1 ? 8 : bt.row_shift;
    k.c_row_shift = bt.row_shift;
    k.result_threshold = bt.result_threshold;
    k.start = bt.start; k.start_nul = bt.start_nul; k.q0 = bt.q0; k.q0_accepting = bt.q0_accepting ? 1 : 0;
    const fx::Literals& L = p->prog.lit;
    k.all_len = (int)L.all.size(); k.pre_len = (int)L.prefix.size(); k.suf_len = (int)L.suffix.size();
    k.all_active = p->prog.literal_only ? 1 : 0;
    k.pre_active = fx::fortran_blank(L.prefix) ? 0 : 1;
    k.suf_active = fx::fortran_blank(L.suffix) ? 0 : 1;
    k.a_table = d.a_table; k.a_classmap = d.a_classmap; k.a_flags = d.a_flags;
    k.a_row_shift = p->has_anchored ? p->anchored.bt.row_shift : 0;
    k.a_start_nul = p->has_anchored ? p->anchored.bt.start_nul : 0;
    k.a_q0 = p->has_anchored ? p->anchored.bt.q0 : 0;
    k.prefix_mode = p->prefix_mode;
    k.steps_left = nullptr;
    p->last_residency = pl.kind == 3 ? FX_TABLE_GLOBAL : FX_TABLE_SMEM;
    p->last_direct = pl.kind <= 1 ? 1 : 0;
    return FX_OK;
}

int check_ready(fx_pattern* p, int op) {
    if (!p) return FX_ERR_BAD_ARGUMENT;
    if (p->prog.status != fx::OK) return p->prog.status;
    if (p->prog.op != op) return FX_ERR_BAD_ARGUMENT;
    return ensure_device(p);
}

template <typename K>
int occupancy_grid(K kernel, int threads, size_t smem, int sm_count, int& blocks_per_sm) {
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
    }
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kernel, threads, smem);
    if (e != cudaSuccess) return cuda_status(e);
    if (blocks_per_sm < 1) return FX_ERR_BAD_ARGUMENT;
    (void)sm_count;
    return FX_OK;
}

// ---- NFA engine (patterns past the eager state cap): parameters and launches ---------------------
void nfa_params(fx_pattern* p, KParams& k, NfaEngine& N) {
    const fx::NfaTables& nt = p->prog.nfa_tables;
    const DeviceTables& d = p->dev;
    memset(&k, 0, sizeof(k));
    const fx::Literals& L = p->prog.lit;
    k.lits = d.lits;
    k.all_len = (int)L.all.size(); k.pre_len = (int)L.prefix.size(); k.suf_len = (int)L.suffix.size();
    k.all_active = p->prog.literal_only ? 1 : 0;
    k.pre_active = fx::fortran_blank(L.prefix) ? 0 : 1;
    k.suf_active = fx::fortran_blank(L.suffix) ? 0 : 1;
    k.q0_accepting = nt.q0_accepting ? 1 : 0;
    N.trans = d.nfa_trans; N.q0 = d.nfa_q0; N.cuts = d.nfa_cuts;
    N.words = nt.words; N.nclasses = nt.nclasses; N.exit_state = nt.exit;
    auto class_of = [&](int cp) { return (int)(std::upper_bound(nt.cuts.begin(), nt.cuts.end(), cp) - nt.cuts.begin()) - 1; };
    N.nul_class = class_of(0); N.ffff_class = class_of(0xFFFF);
    N.q0_accepting = k.q0_accepting;
}
int nfa_grid(fx_pattern* p, int64_t n) {
    long long want = (n + 63) / 64, cap = (long long)p->dev.sm_count * 16;
    int g = (int)(want < cap ? want : cap);
    return g < 1 ? 1 : g;
}
int launch_nfa_bool(fx_pattern* p, int op, const uint8_t* buf, const int64_t* off, int64_t stride, int64_t n, uint8_t* out, cudaStream_t s) {
    if (n <= 0) return n < 0 ? FX_ERR_BAD_ARGUMENT : FX_OK;
    KParams k;
    NfaEngine N;
    nfa_params(p, k, N);
    if (op == FX_OP_MATCH) k_nfa_bool<0><<<nfa_grid(p, n), 64, 0, s>>>(k, N, buf, off, stride, n, out);
    else k_nfa_bool<1><<<nfa_grid(p, n), 64, 0, s>>>(k, N, buf, off, stride, n, out);
    g_launches++;
    return cuda_status(cudaGetLastError());
}
int launch_nfa_regex(fx_pattern* p, const uint8_t* buf, const int64_t* off, int64_t n, int64_t single_len, int64_t* from, int64_t* to,
                     cudaStream_t s) {
    if (n <= 0) return n < 0 ? FX_ERR_BAD_ARGUMENT : FX_OK;
    KParams k;
    NfaEngine N;
    nfa_params(p, k, N);
    k_nfa_regex<<<nfa_grid(p, n), 64, 0, s>>>(k, N, buf, off, n, single_len, from, to);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

// ---- launchers -----------------------------------------------------------------------------
inline size_t staged_bytes(const Plan& pl) { return (size_t)((pl.table_bytes + 15) & ~15); }

template <int OP, int KIND, int VEC>
int launch_fixed_t(fx_pattern* p, const Plan& pl, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out,
                   cudaStream_t s, int generic) {
    auto kern = k_bool_fixed<OP, KIND, VEC>;
    size_t smem = 256 + staged_bytes(pl);
    int bps = 0;
    int rc = occupancy_grid(kern, 256, smem, p->dev.sm_count, bps);
    if (rc) return rc;
    long long want = (n + 255) / 256;
    long long cap = (long long)p->dev.sm_count * bps * 4;   // a few waves, grid-stride inside
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, 256, smem, s>>>(pl.kp, buf, n, stride, out, generic);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

template <int OP, int KIND>
int launch_fixed_v(fx_pattern* p, const Plan& pl, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out,
                   cudaStream_t s, int generic) {
    uintptr_t a = reinterpret_cast<uintptr_t>(buf);
    if (!generic && stride > 0 && stride % 16 == 0 && a % 16 == 0) return launch_fixed_t<OP, KIND, 16>(p, pl, buf, n, stride, out, s, generic);
    if (!generic && stride > 0 && stride % 8 == 0 && a % 8 == 0) return launch_fixed_t<OP, KIND, 8>(p, pl, buf, n, stride, out, s, generic);
    return launch_fixed_t<OP, KIND, 1>(p, pl, buf, n, stride, out, s, generic);
}

// Does every string have to go through the wrapper's literal gates (eval_bool_slow)?  For `.match.` the gates of
// do_matching_exactly compare LENGTHS as well (api_internal_m.F90:199-233: a text equal to the prefix literal matches, a
// text shorter than a literal does not), and those two rules hold for a literal that is blank but not empty (`' +x'`
// has the prefix ' '), which the content compares skip: any non-empty prefix or suffix makes the pattern gated.
// (fx_pattern_info.gated reports this decision; tests/test_host_tables.py checks it against the oracle.)
inline int gated_mode(const fx_pattern* p, int op) {
    const fx::Literals& L = p->prog.lit;
    return (p->prog.literal_only || (op == 0 && (!L.prefix.empty() || !L.suffix.empty())) || (op == 1 && p->prefix_mode == 2)) ? 1 : 0;
}

int launch_sparse(fx_pattern* p, const Plan& pl, const uint8_t* buf, const int64_t* off, int64_t n, int64_t total,
                  uint8_t* out, cudaStream_t s, int64_t stride);

template <int OP>
int launch_fixed(fx_pattern* p, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out, cudaStream_t s) {
    if (n < 0 || stride < 0) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    if (p->prog.nfa_engine) return launch_nfa_bool(p, OP, buf, nullptr, stride, n, out, s);
    Plan pl;
    int rc = make_plan(p, pl);
    if (rc) return rc;
    int generic = gated_mode(p, OP);
    p->last_sparse = 0;
    p->last_compact = 0;
    if (OP == 1 && !generic && p->sparse && stride > 0 && n < (1ll << 31) && env_int("FX_SPARSE", 1)) {   // sparse starts (K2c)
        p->last_sparse = 1;
        return launch_sparse(p, pl, buf, nullptr, n, n * stride, out, s, stride);
    }
    if (pl.kind == 3 && p->compact && !generic && pl.kp.prefix_mode == 0 && stride >= 16 && stride % 16 == 0 &&
        reinterpret_cast<uintptr_t>(buf) % 16 == 0 && env_int("FX_COMPACT", 1)) {       // big automaton, small ASCII alphabet (K1c)
        const bool in_smem = p->residency != FX_TABLE_GLOBAL;
        const size_t smem = 256 + (in_smem ? (size_t)p->prog.bt.nstates * 8 + 16 : 0);
        auto kern_s = k_bool_fixed_compact<OP, true>;
        auto kern_g = k_bool_fixed_compact<OP, false>;
        int bps = 0;
        int rc2 = in_smem ? occupancy_grid(kern_s, 1024, smem, p->dev.sm_count, bps) : occupancy_grid(kern_g, 1024, smem, p->dev.sm_count, bps);
        if (rc2) return rc2;
        long long want = (n + 1023) / 1024, cap = (long long)p->dev.sm_count * bps * 2;
        const int grid = (int)(want < cap ? want : cap);
        if (in_smem) kern_s<<<grid, 1024, smem, s>>>(pl.kp, p->dev.ctab4, p->dev.cmap4, buf, n, stride, out);
        else kern_g<<<grid, 1024, smem, s>>>(pl.kp, p->dev.ctab4, p->dev.cmap4, buf, n, stride, out);
        g_launches++;
        p->last_compact = in_smem ? 1 : 2;
        p->last_residency = in_smem ? FX_TABLE_SMEM : FX_TABLE_GLOBAL;
        return cuda_status(cudaGetLastError());
    }
    if (pl.kind == 0) return launch_fixed_v<OP, 0>(p, pl, buf, n, stride, out, s, generic);
    if (pl.kind == 2) return launch_fixed_v<OP, 2>(p, pl, buf, n, stride, out, s, generic);
    return launch_fixed_v<OP, 3>(p, pl, buf, n, stride, out, s, generic);
}

// tiles of `spt` consecutive strings; up to `cap` bytes of a tile's text are staged in shared memory.  The tile is
// sized so that 4 CTAs fit one SM's shared memory (227 KB usable, 1 KB reserved per CTA).
struct Tiling {
    int spt, cap;
    int64_t ntiles;
    int table_smem;  // staged table bytes, 16-byte rounded
    size_t smem;
};

Tiling make_tiling(const Plan& pl, int64_t n, int64_t total, int extra = 0, int64_t max_cap = 1 << 30) {
    Tiling t;
    int64_t avg = n > 0 ? (total + n - 1) / n : 1;
    if (avg < 1) avg = 1;
    t.table_smem = (int)staged_bytes(pl);
    const int64_t per_cta = (227 * 1024) / 4 - 1024;
    // strings per tile: about one per thread, fewer when strings are long, more when they are short
    int64_t spt = 0, cap = 0;
    for (int iter = 0; iter < 2; iter++) {
        int64_t fixed = tile_offset(t.table_smem, (int)(spt ? spt : 256)) + 64 + 128 + extra;
        cap = per_cta - fixed;
        if (cap < 8192) cap = 8192;
        if (cap > max_cap) cap = max_cap;
        cap &= ~(int64_t)127;
        spt = (cap * 4 / 5) / avg;           // expect the tile to fill ~80 % of the staged capacity
        spt = (spt / 32) * 32;
        if (spt < 32) spt = 32;
        if (spt > 2048) spt = 2048;
    }
    t.spt = (int)spt;
    t.cap = (int)cap;
    t.ntiles = (n + spt - 1) / spt;
    t.smem = (size_t)tile_offset(t.table_smem, t.spt) + (size_t)extra + (size_t)t.cap + 64;
    return t;
}

template <int OP, int KIND>
int launch_ragged_t(fx_pattern* p, const Plan& pl, const uint8_t* buf, const int64_t* off, int64_t n, int64_t total,
                    uint8_t* out, cudaStream_t s, int generic) {
    auto kern = k_bool_ragged<OP, KIND>;
    Tiling t = make_tiling(pl, n, total);
    int bps = 0;
    int rc = occupancy_grid(kern, 256, t.smem, p->dev.sm_count, bps);
    if (rc) return rc;
    long long cap = (long long)p->dev.sm_count * bps;
    int grid = (int)(t.ntiles < cap ? t.ntiles : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, 256, t.smem, s>>>(pl.kp, buf, off, n, total, out, t.spt, t.cap, t.ntiles, t.table_smem, generic);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

// K2c: a warp sweeps tiles of `spt` consecutive strings, about 24 KB of text each
template <int KIND, int NR, bool HIGH, bool TWO>
int launch_sparse_t(fx_pattern* p, const Plan& pl, const SparseParams& sp, int table_bytes, const uint8_t* buf,
                    const int64_t* off, int64_t n, int64_t total, uint8_t* out, cudaStream_t s, int64_t stride) {
    auto kern = k_in_sparse<KIND, NR, HIGH, TWO>;
    int64_t avg = n > 0 ? (total + n - 1) / n : 1;
    if (avg < 1) avg = 1;
    int64_t want = (24 * 1024) / avg;       // (one sweep segment holds 32 KB)
    const int spt = (int)(want < 32 ? 32 : want > 4096 ? 4096 : want);
    const int64_t ntiles = (n + spt - 1) / spt;
    const int table_smem = KIND == 3 ? 0 : (table_bytes + 15) & ~15;
    const size_t smem = (size_t)sparse_shared_head(table_smem) + 8 * (size_t)SPARSE_WARP_BYTES;
    int bps = 0;
    int rc = occupancy_grid(kern, 256, smem, p->dev.sm_count, bps);
    if (rc) return rc;
    long long cap = (long long)p->dev.sm_count * bps;
    long long wantg = (ntiles + 7) / 8;
    int grid = (int)(wantg < cap ? wantg : cap);
    if (grid < 1) grid = 1;
    // a pattern that neither accepts the empty text nor starts on the leading NUL decides no string in the per-string
    // phase: every result is "false unless a start wins", so the results are cleared here, at copy speed
    const int prezeroed = sp.start_nul == 0 && pl.kp.q0_accepting == 0;
    if (prezeroed) CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)n, s));
    kern<<<grid, 256, smem, s>>>(pl.kp, sp, buf, off, n, total, out, spt, ntiles, table_smem, prezeroed, stride);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

template <int KIND, bool HIGH>
int launch_sparse_k(fx_pattern* p, const Plan& pl, const SparseParams& sp, int tb, const uint8_t* buf, const int64_t* off,
                    int64_t n, int64_t total, uint8_t* out, cudaStream_t s, int64_t stride) {
    if (p->first.sweep_nr == 1 && p->first.sweep_lo[0] == p->first.sweep_hi[0]) {      // one byte value: the cheaper zero-byte test
        const SparseParams& one = sp;      // (fill_sweep has put the byte value into add_lo[0])
        if (p->first.two) return launch_sparse_t<KIND, -1, HIGH, true>(p, pl, one, tb, buf, off, n, total, out, s, stride);
        return launch_sparse_t<KIND, -1, HIGH, false>(p, pl, one, tb, buf, off, n, total, out, s, stride);
    }
    switch (p->first.sweep_nr) {
        case 0: return launch_sparse_t<KIND, 0, true, false>(p, pl, sp, tb, buf, off, n, total, out, s, stride);
        case 1: return launch_sparse_t<KIND, 1, HIGH, false>(p, pl, sp, tb, buf, off, n, total, out, s, stride);
        case 2: return launch_sparse_t<KIND, 2, HIGH, false>(p, pl, sp, tb, buf, off, n, total, out, s, stride);
        case 3: return launch_sparse_t<KIND, 3, HIGH, false>(p, pl, sp, tb, buf, off, n, total, out, s, stride);
        default: return launch_sparse_t<KIND, 4, HIGH, false>(p, pl, sp, tb, buf, off, n, total, out, s, stride);
    }
}

void fill_sweep(const FirstSet& f, SparseParams& sp) {
    for (int r = 0; r < 4; r++) {
        const int k = r < f.sweep_nr ? r : 0;       // unused slots repeat range 0
        sp.add_lo[r] = (0x80u - f.sweep_lo[k]) * 0x01010101u;
        sp.add_hi[r] = (0x7Fu - f.sweep_hi[k]) * 0x01010101u;
    }
    if (f.sweep_nr == 1 && f.sweep_lo[0] == f.sweep_hi[0]) sp.add_lo[0] = f.sweep_lo[0] * 0x01010101u;   // NR = -1 form
    sp.second = f.second * 0x01010101u;
    sp.second_high = f.second_high ? 0xFFFFFFFFu : 0u;
}

int launch_sparse(fx_pattern* p, const Plan& pl, const uint8_t* buf, const int64_t* off, int64_t n, int64_t total,
                  uint8_t* out, cudaStream_t s, int64_t stride) {
    const fx::ByteTable& at = p->anchored.bt;
    const DeviceTables& d = p->dev;
    SparseParams sp;
    sp.table = d.a_table; sp.classmap = d.a_classmap; sp.flags = d.a_flags;
    sp.table_words = (int)at.table.size();
    sp.row_shift = at.row_shift;
    sp.q0 = at.q0; sp.start_nul = at.start_nul;
    fill_sweep(p->first, sp);
    const int tb = (int)at.table.size() * 2;
    const bool smem_table = p->residency != FX_TABLE_GLOBAL && tb <= 24 * 1024;
    if (smem_table)
        return p->first.high ? launch_sparse_k<2, true>(p, pl, sp, tb, buf, off, n, total, out, s, stride)
                             : launch_sparse_k<2, false>(p, pl, sp, tb, buf, off, n, total, out, s, stride);
    return p->first.high ? launch_sparse_k<3, true>(p, pl, sp, tb, buf, off, n, total, out, s, stride)
                         : launch_sparse_k<3, false>(p, pl, sp, tb, buf, off, n, total, out, s, stride);
}

template <int OP>
int launch_ragged(fx_pattern* p, const uint8_t* buf, const int64_t* off, int64_t n, int64_t total, uint8_t* out,
                  cudaStream_t s) {
    if (n < 0 || total < 0) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    if (p->prog.nfa_engine) return launch_nfa_bool(p, OP, buf, off, 0, n, out, s);
    Plan pl;
    int rc = make_plan(p, pl);
    if (rc) return rc;
    int generic = gated_mode(p, OP);
    p->last_sparse = 0;
    if (OP == 1 && !generic && p->sparse && n < (1ll << 31) && env_int("FX_SPARSE", 1)) {      // sparse starts (K2c)
        p->last_sparse = 1;
        return launch_sparse(p, pl, buf, off, n, total, out, s, 0);
    }
    if (pl.kind == 0) return launch_ragged_t<OP, 0>(p, pl, buf, off, n, total, out, s, generic);
    if (pl.kind == 2) return launch_ragged_t<OP, 2>(p, pl, buf, off, n, total, out, s, generic);
    return launch_ragged_t<OP, 3>(p, pl, buf, off, n, total, out, s, generic);
}

template <int KIND>
int launch_regex_ragged_t(fx_pattern* p, const Plan& pl, const uint8_t* buf, const int64_t* off, int64_t n,
                          int64_t total, int64_t* from, int64_t* to, cudaStream_t s) {
    auto kern = k_regex_ragged<KIND>;
    Tiling t = make_tiling(pl, n, total);
    int bps = 0;
    int rc = occupancy_grid(kern, 256, t.smem, p->dev.sm_count, bps);
    if (rc) return rc;
    long long cap = (long long)p->dev.sm_count * bps;
    int grid = (int)(t.ntiles < cap ? t.ntiles : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, 256, t.smem, s>>>(pl.kp, buf, off, n, total, from, to, t.spt, t.cap, t.ntiles, t.table_smem);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

// fills the parameter block of the linear-time span path (K3f, and the long-buffer state-map scan)
void fill_span_params(fx_pattern* p, SpanParams& sp) {
    const fx::ByteTable& st = p->prog.span_bt;
    const fx::RevAutomaton& rv = p->prog.rev;
    const DeviceTables& d = p->dev;
    sp.direct = d.sp_direct; sp.table = d.sp_table; sp.classmap = d.sp_classmap; sp.endinfo = d.sp_endinfo;
    sp.nstates = st.nstates; sp.row_shift = st.row_shift; sp.start = st.start;
    sp.start_acc = (st.flags[(size_t)st.start] & fxk::SF_ACC) ? 1 : 0;
    sp.rdelta = d.r_delta; sp.rpage = d.r_page; sp.rmixed = d.r_mixed; sp.cuts = d.r_cuts;
    sp.rstates = rv.nstates; sp.rclasses = rv.nclasses; sp.rstart = rv.start;
    sp.nul_class = p->prog.span_cp.class_of(0);
    sp.ffff_class = p->prog.span_cp.class_of(0xFFFF);
    sp.nmixed = (int)(rv.mixed.size() / 64);
}

template <int FK, bool RS>
int launch_span_t(fx_pattern* p, const Plan& pl, const SpanParams& sp, int fwd_bytes, const uint8_t* buf,
                  const int64_t* off, int64_t n, int64_t total, int64_t* from, int64_t* to, cudaStream_t s) {
    auto kern = k_span_ragged<FK, RS>;
    // one CTA of SPAN_WARPS warps per SM; every warp stages its own tiles: the tables take their share of the SM's
    // shared memory once, the rest is divided among the warps
    int64_t avg = n > 0 ? (total + n - 1) / n : 1;
    if (avg < 1) avg = 1;
    const SpanHead H = span_head(fwd_bytes, sp.rstates * sp.rclasses * 2, sp.nmixed, RS);
    int per_warp = ((227 * 1024 - 1024 - H.bytes) / SPAN_WARPS) & ~127;
    if (per_warp < 1024) return FX_ERR_BAD_ARGUMENT;
    int cap = per_warp, spt = 1;
    for (;;) {
        int64_t want = ((int64_t)cap * 7 / 8) / avg;       // expect the tile to fill most of the staged capacity
        spt = (int)(want < 1 ? 1 : want > 512 ? 512 : want);
        if (cap <= 512 || span_layout(spt, cap).warp_bytes <= per_warp) break;
        cap -= 128;
    }
    while (spt > 1 && span_layout(spt, cap).warp_bytes > per_warp) spt--;
    const int64_t ntiles = (n + spt - 1) / spt;
    const size_t smem = (size_t)H.bytes + (size_t)SPAN_WARPS * (size_t)span_layout(spt, cap).warp_bytes;
    int bps = 0;
    int rc = occupancy_grid(kern, SPAN_WARPS * 32, smem, p->dev.sm_count, bps);
    if (rc) return rc;
    long long capg = (long long)p->dev.sm_count * bps;
    long long want = (ntiles + SPAN_WARPS - 1) / SPAN_WARPS;
    int grid = (int)(want < capg ? want : capg);
    if (grid < 1) grid = 1;
    kern<<<grid, SPAN_WARPS * 32, smem, s>>>(pl.kp, sp, buf, off, n, total, from, to, spt, cap, ntiles, fwd_bytes);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

int launch_regex_ragged(fx_pattern* p, const uint8_t* buf, const int64_t* off, int64_t n, int64_t total,
                        int64_t* from, int64_t* to, cudaStream_t s) {
    if (n < 0 || total < 0) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    if (p->prog.nfa_engine) return launch_nfa_regex(p, buf, off, n, 0, from, to, s);
    Plan pl;
    int rc = make_plan(p, pl);
    if (rc) return rc;
    if (p->prog.has_span && env_int("FX_SPAN_LINEAR", 1)) {       // linear-time span path (K3f)
        const fx::ByteTable& st = p->prog.span_bt;
        const fx::RevAutomaton& rv = p->prog.rev;
        SpanParams sp;
        fill_span_params(p, sp);
        const int classed_bytes = (int)st.table.size() * 2;
        int fk = p->residency == FX_TABLE_GLOBAL ? 2 : p->dev.sp_direct ? 0 : classed_bytes <= SPAN_CLASSED_SMEM_BYTES ? 1 : 2;
        fk = env_int("FX_SPAN_FK", fk);
        if (fk == 0 && !p->dev.sp_direct) fk = 1;
        const int fwd_bytes = fk == 0 ? st.nstates * SPAN_ROW * 2 : fk == 1 ? classed_bytes : 0;
        const bool rs = !rv.page.empty() && (int)(rv.delta16.size() * 2 + 1024 + rv.mixed.size()) <= SPAN_REV_SMEM_BYTES;
        if (fk == 0) return rs ? launch_span_t<0, true>(p, pl, sp, fwd_bytes, buf, off, n, total, from, to, s)
                               : launch_span_t<0, false>(p, pl, sp, fwd_bytes, buf, off, n, total, from, to, s);
        if (fk == 1) return rs ? launch_span_t<1, true>(p, pl, sp, fwd_bytes, buf, off, n, total, from, to, s)
                               : launch_span_t<1, false>(p, pl, sp, fwd_bytes, buf, off, n, total, from, to, s);
        return rs ? launch_span_t<2, true>(p, pl, sp, fwd_bytes, buf, off, n, total, from, to, s)
                  : launch_span_t<2, false>(p, pl, sp, fwd_bytes, buf, off, n, total, from, to, s);
    }
    if (pl.kind == 1) return launch_regex_ragged_t<1>(p, pl, buf, off, n, total, from, to, s);
    if (pl.kind == 2) return launch_regex_ragged_t<2>(p, pl, buf, off, n, total, from, to, s);
    return launch_regex_ragged_t<3>(p, pl, buf, off, n, total, from, to, s);
}

template <int KIND>
int launch_scan_t(fx_pattern* p, const Plan& pl, const uint8_t* buf, const ScanWindow& W, unsigned long long* best,
                  cudaStream_t s, const unsigned long long* gate, const unsigned long long* run_if) {
    auto kern = k_buffer_scan<KIND>;
    int table_smem = (int)staged_bytes(pl);
    size_t smem = (size_t)scan_smem_bytes(table_smem);
    int bps = 0;
    int rc = occupancy_grid(kern, 256, smem, p->dev.sm_count, bps);
    if (rc) return rc;
    long long units = ((W.start_hi - W.start_lo) >> 4) + 1;
    long long want = (units + 255) / 256;
    long long cap = (long long)p->dev.sm_count * bps;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, 256, smem, s>>>(pl.kp, buf, W, best, table_smem, gate, run_if);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

template <int KIND, int NR, bool HIGH, bool PREFIX>
int launch_scan_sparse_t(fx_pattern* p, const Plan& pl, const SparseParams& sp, const uint8_t* buf, const ScanWindow& W,
                         unsigned long long* best, cudaStream_t s, const unsigned long long* gate,
                         const unsigned long long* run_if, ScanBudget budget) {
    auto kern = k_buffer_scan_sparse<KIND, NR, HIGH, PREFIX>;
    int table_smem = (int)staged_bytes(pl);
    size_t smem = (size_t)scan_sparse_smem_bytes(table_smem);
    int bps = 0;
    int rc = occupancy_grid(kern, 256, smem, p->dev.sm_count, bps);
    if (rc) return rc;
    long long groups = ((W.start_hi - W.start_lo) >> 12) + 1;       // 4 KB per warp and step
    long long want = (groups + 7) / 8;
    long long cap = (long long)p->dev.sm_count * bps;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, 256, smem, s>>>(pl.kp, sp, buf, W, best, table_smem, gate, run_if, budget);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

template <int KIND>
int launch_scan_sparse(fx_pattern* p, const Plan& pl, const uint8_t* buf, const ScanWindow& W, unsigned long long* best,
                       cudaStream_t s, const unsigned long long* gate, const unsigned long long* run_if, ScanBudget bg) {
    SparseParams sp;
    memset(&sp, 0, sizeof(sp));
    fill_sweep(p->first, sp);
    const FirstSet& f = p->first;
    const bool one = f.sweep_nr == 1 && f.sweep_lo[0] == f.sweep_hi[0];
    if (f.sweep_nr == 0) return launch_scan_sparse_t<KIND, 0, true, false>(p, pl, sp, buf, W, best, s, gate, run_if, bg);
    if (one) return f.high ? launch_scan_sparse_t<KIND, -1, true, false>(p, pl, sp, buf, W, best, s, gate, run_if, bg)
                           : launch_scan_sparse_t<KIND, -1, false, false>(p, pl, sp, buf, W, best, s, gate, run_if, bg);
    if (f.sweep_nr == 1) return f.high ? launch_scan_sparse_t<KIND, 1, true, false>(p, pl, sp, buf, W, best, s, gate, run_if, bg)
                                       : launch_scan_sparse_t<KIND, 1, false, false>(p, pl, sp, buf, W, best, s, gate, run_if, bg);
    return f.high ? launch_scan_sparse_t<KIND, 2, true, false>(p, pl, sp, buf, W, best, s, gate, run_if, bg)
                  : launch_scan_sparse_t<KIND, 2, false, false>(p, pl, sp, buf, W, best, s, gate, run_if, bg);
}

// candidates = the occurrences of the prefix literal: sweep for its first byte
template <int KIND>
int launch_scan_prefix(fx_pattern* p, const Plan& pl, const uint8_t* buf, const ScanWindow& W, unsigned long long* best,
                       cudaStream_t s, const unsigned long long* run_if, ScanBudget bg) {
    SparseParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.add_lo[0] = (unsigned char)p->prog.lit.prefix[0] * 0x01010101u;      // NR = -1 form
    return launch_scan_sparse_t<KIND, -1, false, true>(p, pl, sp, buf, W, best, s, nullptr, run_if, bg);
}

// scan starts [start_lo, start_hi) of a window; d_best[0] (min key), d_best[1] (undecided attempts) and d_best[2]
// (prefix occurrences seen) must have been initialised by the caller.
//   mode SCAN_AUTO   the pattern's own candidates: the occurrences of its prefix literal if it has one, else every
//                    character boundary
//   mode SCAN_ALL    every character boundary, whatever the pattern (what the reference does when the prefix occurs
//                    nowhere in the text); `gate`, if given, cancels the launch when *gate != 0
enum { SCAN_AUTO = 0, SCAN_ALL = 1 };
int launch_scan(fx_pattern* p, const uint8_t* buf, const ScanWindow& W, unsigned long long* best, cudaStream_t s,
                int mode = SCAN_AUTO, const unsigned long long* gate = nullptr, const unsigned long long* run_if = nullptr,
                ScanBudget bg = ScanBudget{nullptr, nullptr, 0ull}) {
    if (W.len < 0 || W.start_lo < 0 || W.start_hi > W.len || W.start_lo > W.start_hi) return FX_ERR_BAD_ARGUMENT;
    if (p->prog.nfa_engine) return FX_ERR_DFA_STATE_CAP;        // the window forms need the table engine
    const bool prefixed = p->prog.prefix_active && !p->prog.literal_only;
    // a prefix whose occurrences can overlap, or a non-empty suffix, make the candidate list sequential: not handled
    if (prefixed && !p->prefix_scan) return FX_ERR_PREFILTER_UNSUPPORTED;
    Plan pl;
    int rc = make_plan(p, pl);
    if (rc) return rc;
    if (W.start_lo == W.start_hi) return FX_OK;
    p->last_sparse = 0;
    if (pl.kp.all_active) {          // the pattern is one literal: parallel index() (K4L)
        SparseParams sp;
        memset(&sp, 0, sizeof(sp));
        sp.add_lo[0] = (unsigned char)p->prog.lit.all[0] * 0x01010101u;      // NR = -1 form
        long long groups = ((W.start_hi - W.start_lo) >> 12) + 1;
        long long want = (groups + 7) / 8, cap = (long long)p->dev.sm_count * 8;
        int grid = (int)(want < cap ? want : cap);
        k_buffer_literal<<<grid < 1 ? 1 : grid, 256, 0, s>>>(pl.kp.lits, pl.kp.all_len, sp, buf, W, best);
        g_launches++;
        return cuda_status(cudaGetLastError());
    }
    if (prefixed && mode == SCAN_AUTO) {
        if (pl.kind == 1) return launch_scan_prefix<1>(p, pl, buf, W, best, s, run_if, bg);
        if (pl.kind == 2) return launch_scan_prefix<2>(p, pl, buf, W, best, s, run_if, bg);
        return launch_scan_prefix<3>(p, pl, buf, W, best, s, run_if, bg);
    }
    if (p->sparse && p->first.sweep_nr <= 2 && env_int("FX_SPARSE", 1)) {     // SWAR first-byte filter
        p->last_sparse = 1;
        if (pl.kind == 1) return launch_scan_sparse<1>(p, pl, buf, W, best, s, gate, run_if, bg);
        if (pl.kind == 2) return launch_scan_sparse<2>(p, pl, buf, W, best, s, gate, run_if, bg);
        return launch_scan_sparse<3>(p, pl, buf, W, best, s, gate, run_if, bg);
    }
    if (pl.kind == 1) return launch_scan_t<1>(p, pl, buf, W, best, s, gate, run_if);
    if (pl.kind == 2) return launch_scan_t<2>(p, pl, buf, W, best, s, gate, run_if);
    return launch_scan_t<3>(p, pl, buf, W, best, s, gate, run_if);
}

int launch_finish(fx_pattern* p, const uint8_t* buf, const ScanWindow& W, const unsigned long long* best,
                  int64_t* from_to, int whole_text, cudaStream_t s, const unsigned long long* done = nullptr,
                  const unsigned long long* use_alt = nullptr, const unsigned long long* best_alt = nullptr,
                  const unsigned long long* spent = nullptr) {
    if (p->prog.nfa_engine) return FX_ERR_DFA_STATE_CAP;
    Plan pl;
    int rc = make_plan(p, pl);
    if (rc) return rc;
    k_buffer_finish<<<1, 1, 0, s>>>(pl.kp, buf, W, best, from_to, whole_text, done, use_alt, best_alt, spent);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

// ---- the long-buffer search: work area layout (64-bit words) -----------------------------------------------
//   [0] smallest winning start (key), [1] undecided attempts, [2] prefix occurrences      -- K4, first run
//   [4] 1 = K4 spent its work budget (or was not tried): the state-map scan runs           [5] K4's step counter
//   [6] state-map scan: end of the match, [7] its status (1 = declined)
//   [8] 1 = the state-map scan has written the answer        [9] 1 = it declined: K4 runs again, without a budget
//   [12..14] key / undecided / occurrences of that second run
//   [16..17] presence flags of the prefix / suffix literal (sequential candidate list)
//   [24..28] fx_regex_buffer_all_dev: the loop's state (rest, count, done, far step wanted, work budget spent)
//   [30..31] fx_regex_buffer_all_dev: from_to of a far step
//   from byte 4096: the region maps of the state-map scan (rc, re: 32 x u16 per region; rl: 32 x i64 per region)
constexpr size_t WORK_HEAD = 4096;
constexpr int64_t SM_SEG = 32 * (int64_t)SM_SUB;                // one segment: 32 lanes x SM_SUB bytes
inline int64_t statemap_max_regions(int64_t len) {
    int64_t r = len / SM_SEG + 2;
    return r > 65536 ? 65536 : r;
}
inline size_t buffer_work_bytes(int64_t len) { return WORK_HEAD + (size_t)statemap_max_regions(len < 0 ? 0 : len) * 32 * 12 + 256; }

template <int FK>
int launch_statemap_t(fx_pattern* p, const SpanParams& sp, StateMapParams mp, int fwd_bytes, const uint8_t* buf, int64_t len,
                      cudaStream_t s, const unsigned long long* run_if, bool window) {
    auto kern = window ? k_statemap_regions<FK, true> : k_statemap_regions<FK, false>;
    const size_t smem = (size_t)((256 + fwd_bytes + 15) & ~15) + 256 * (1 + SM_M) * 2 + 256 + SM_WARPS * 32 * sizeof(SubMap) + SM_WARPS * 32 * 2 + 64;
    int bps = 0;
    int rc = occupancy_grid(kern, SM_WARPS * 32, smem, p->dev.sm_count, bps);
    if (rc) return rc;
    // regions: about four per resident warp, whole segments, at most what the work area holds
    const int64_t nwarps = (int64_t)p->dev.sm_count * bps * SM_WARPS;
    int64_t region = (len + nwarps * 4 - 1) / (nwarps * 4);
    region = (region + SM_SEG - 1) / SM_SEG * SM_SEG;
    if (region < SM_SEG) region = SM_SEG;
    const int64_t cap = statemap_max_regions(len);
    while ((len + 15 + region - 1) / region > cap) region += SM_SEG;
    mp.region_bytes = region;
    mp.nregions = (len + 15 + region - 1) / region;
    if (mp.nregions < 1) mp.nregions = 1;
    long long want = (mp.nregions + SM_WARPS - 1) / SM_WARPS, capg = (long long)p->dev.sm_count * bps;
    int grid = (int)(want < capg ? want : capg);
    kern<<<grid < 1 ? 1 : grid, SM_WARPS * 32, smem, s>>>(sp, mp, buf, len, fwd_bytes, run_if);
    g_launches++;
    rc = cuda_status(cudaGetLastError());
    if (rc) return rc;
    if (window) k_statemap_compose<true><<<1, 1024, 0, s>>>(sp, mp, len, run_if);
    else k_statemap_compose<false><<<1, 1024, 0, s>>>(sp, mp, len, run_if);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

// the region and compose kernels of the state-map scan over buf[0, len), region maps in `work`.  back / pos0: see
// StateMapParams (0 / 0 for a whole text); `result`: 2 words, or the slab map of the window form (window = true)
int launch_statemap_scan(fx_pattern* p, const SpanParams& sp, const uint8_t* buf, int64_t len, int64_t back, int64_t pos0,
                         unsigned long long* work, long long* result, cudaStream_t s, const unsigned long long* run_if, bool window) {
    const fx::ByteTable& st = p->prog.span_bt;
    StateMapParams mp;
    mp.reach = p->dev.sm_reach; mp.img = p->dev.sm_img; mp.sync = p->dev.sm_sync; mp.nreach = (int)p->sm_reach.size();
    uint8_t* maps = reinterpret_cast<uint8_t*>(work) + WORK_HEAD;
    const int64_t cap = statemap_max_regions(len);
    mp.rc = reinterpret_cast<uint16_t*>(maps);
    mp.re = mp.rc + cap * 32;
    mp.rl = reinterpret_cast<long long*>(maps + (size_t)cap * 32 * 4);
    mp.result = result;
    mp.region_bytes = 0; mp.nregions = 0;
    mp.back = back; mp.pos0 = pos0;
    const int classed_bytes = (int)st.table.size() * 2;
    int fk = p->residency == FX_TABLE_GLOBAL ? 2 : p->dev.sp_direct ? 0 : classed_bytes <= SPAN_CLASSED_SMEM_BYTES ? 1 : 2;
    fk = env_int("FX_SPAN_FK", fk);
    if (fk == 0 && !p->dev.sp_direct) fk = 1;
    const int fwd_bytes = fk == 0 ? st.nstates * SPAN_ROW * 2 : fk == 1 ? classed_bytes : 0;
    return fk == 0 ? launch_statemap_t<0>(p, sp, mp, fwd_bytes, buf, len, s, run_if, window)
         : fk == 1 ? launch_statemap_t<1>(p, sp, mp, fwd_bytes, buf, len, s, run_if, window)
                   : launch_statemap_t<2>(p, sp, mp, fwd_bytes, buf, len, s, run_if, window);
}

// the state-map scan + its finish, gated on *run_if != 0 (nullptr: always)
int launch_statemap(fx_pattern* p, const uint8_t* buf, int64_t len, int64_t* from_to, unsigned long long* work, cudaStream_t s,
                    const unsigned long long* run_if) {
    SpanParams sp;
    fill_span_params(p, sp);
    long long* result = reinterpret_cast<long long*>(work + 6);
    int rc = launch_statemap_scan(p, sp, buf, len, 0, 0, work, result, s, run_if, false);
    if (rc) return rc;
    // with a prefix literal the answer only stands if the winner begins with the literal's own bytes (see launch_buffer)
    const bool check = p->prog.prefix_active && !p->prog.literal_only;
    k_buffer_finish_span<<<1, 1, 0, s>>>(sp, buf, len, result, from_to, work + 8, work + 9, run_if,
                                         check ? p->dev.lits + p->prog.lit.all.size() : nullptr, check ? (int)p->prog.lit.prefix.size() : 0);
    g_launches++;
    return cuda_status(cudaGetLastError());
}

int launch_buffer(fx_pattern* p, const uint8_t* buf, int64_t len, int64_t* from_to, unsigned long long* work,
                  cudaStream_t s) {
    if (len < 0) return FX_ERR_BAD_ARGUMENT;
    if (p->prog.nfa_engine)          // one thread walks the buffer with the reference's own loop: defined, not fast
        return launch_nfa_regex(p, buf, nullptr, 1, len, from_to, from_to + 1, s);
    CUDA_TRY(cudaMemsetAsync(work, 0, 128, s));
    CUDA_TRY(cudaMemsetAsync(work, 0xFF, 8, s));
    CUDA_TRY(cudaMemsetAsync(work + 12, 0xFF, 8, s));
    unsigned long long* best = work;
    ScanWindow W{len, 0, len, 0, 1, 1};
    const bool prefixed = p->prog.prefix_active && !p->prog.literal_only;
    p->last_statemap = 0;
    if (prefixed && !p->prefix_scan) {           // sequential candidate list (bordered prefix / suffix literal): one thread, exact
        Plan pl;
        int rc = make_plan(p, pl);
        if (rc) return rc;
        // parallel presence sweeps for the two literals first: "prefix somewhere, suffix nowhere" is an immediate no-match
        const fx::Literals& L = p->prog.lit;
        const bool quick = pl.kp.suf_active && pl.kp.pre_active && len >= 1 && L.prefix.find('\0') == std::string::npos &&
                           L.suffix.find('\0') == std::string::npos;
        if (quick) {
            CUDA_TRY(cudaMemsetAsync(work + 16, 0xFF, 16, s));
            long long groups = (len >> 12) + 1, want = (groups + 7) / 8, cap = (long long)p->dev.sm_count * 8;
            const int grid = (int)(want < cap ? want : cap);
            SparseParams sp;
            memset(&sp, 0, sizeof(sp));
            sp.add_lo[0] = (unsigned char)L.prefix[0] * 0x01010101u;
            k_buffer_literal<<<grid, 256, 0, s>>>(pl.kp.lits + pl.kp.all_len, pl.kp.pre_len, sp, buf, W, work + 16);
            sp.add_lo[0] = (unsigned char)L.suffix[0] * 0x01010101u;
            k_buffer_literal<<<grid, 256, 0, s>>>(pl.kp.lits + pl.kp.all_len + pl.kp.pre_len, pl.kp.suf_len, sp, buf, W, work + 17);
            g_launches += 2;
        }
        k_buffer_sequential<<<1, 1, 0, s>>>(pl.kp, buf, len, from_to, quick ? work + 16 : nullptr, quick ? work + 17 : nullptr);
        g_launches++;
        return cuda_status(cudaGetLastError());
    }
    // Patterns with a linear-time span path: the candidate-start scan (K4) is the fast path when candidates are rare
    // (sparse first-byte set) -- under a work budget; past the budget, and for every other such pattern, the chunked
    // state-map scan (K5) answers in linear time; should that scan decline (too many states can arrive at a region
    // boundary), K4 runs without a budget.  All gating is on device flags: no host round trip.
    const int sm_mode = env_int("FX_STATEMAP", 1);             // 0 off, 1 as described, 2 always the state-map scan
    const bool sm_ok = p->statemap && !p->prog.literal_only && !prefixed && len >= 2 && sm_mode != 0;
    if (prefixed && p->statemap && p->prefix_neutral && len >= 2 && sm_mode != 0) {
        // A prefix literal: Forgex's candidates are the literal's occurrences (every boundary when it occurs nowhere).
        // `a.*b` over a megabyte of `a` makes that quadratic too.  Same remedy: the candidate scan runs under the work
        // budget; past it the state-map scan answers -- it tries EVERY boundary, which is the same answer whenever the
        // winner begins with the literal's own bytes (the prefilter is provably neutral for this pattern: every match
        // begins with the literal's code points; only an overlong encoding of them could differ).  If the winner does
        // not, or the scan declines, the candidate scan runs again without a budget.
        ScanBudget bg{work + 5, work + 4, (unsigned long long)len * 16ull + (4ull << 20)};
        int rc = sm_mode == 2 ? FX_OK : launch_scan(p, buf, W, best, s, SCAN_AUTO, nullptr, nullptr, bg);
        if (rc) return rc;
        if (sm_mode == 2) CUDA_TRY(cudaMemsetAsync(work + 4, 0x01, 1, s));
        else if ((rc = launch_scan(p, buf, W, best, s, SCAN_ALL, best + 2, nullptr, bg))) return rc;
        if ((rc = launch_statemap(p, buf, len, from_to, work, s, work + 4))) return rc;
        if ((rc = launch_scan(p, buf, W, work + 12, s, SCAN_AUTO, nullptr, work + 9))) return rc;
        if ((rc = launch_scan(p, buf, W, work + 12, s, SCAN_ALL, work + 14, work + 9))) return rc;
        p->last_statemap = sm_mode == 2 ? 1 : 2;
        return launch_finish(p, buf, W, best, from_to, 1, s, work + 8, work + 9, work + 12);
    }
    if (sm_ok) {
        const bool k4_first = p->sparse && p->first.sweep_nr <= 2 && env_int("FX_SPARSE", 1) && sm_mode != 2;
        int rc;
        if (k4_first) {
            ScanBudget bg{work + 5, work + 4, (unsigned long long)len * 16ull + (4ull << 20)};
            rc = launch_scan(p, buf, W, best, s, SCAN_AUTO, nullptr, nullptr, bg);
            if (rc) return rc;
        } else {
            CUDA_TRY(cudaMemsetAsync(work + 4, 0x01, 1, s));  // no budgeted run: straight to the state-map scan
        }
        rc = launch_statemap(p, buf, len, from_to, work, s, work + 4);
        if (rc) return rc;
        rc = launch_scan(p, buf, W, work + 12, s, SCAN_AUTO, nullptr, work + 9);      // only if the state-map scan declined
        if (rc) return rc;
        p->last_statemap = k4_first ? 2 : 1;
        return launch_finish(p, buf, W, best, from_to, 1, s, work + 8, work + 9, work + 12);
    }
    // What is left: patterns without the span path (a cap was passed), and prefix literals that are not provably neutral.
    // The candidate scan still runs under the work budget; without a linear-time stand-in a spent budget is reported as
    // (-2, -2) = FX_ERR_WORK_BUDGET instead of occupying the GPU with the reference's quadratic loop.
    ScanBudget bg{work + 5, work + 4, (unsigned long long)len * 16ull + (4ull << 20)};
    const bool budgeted = env_int("FX_STATEMAP", 1) != 0;
    if (!budgeted) bg = ScanBudget{nullptr, nullptr, 0ull};
    if (len >= 1) {
        int rc = launch_scan(p, buf, W, best, s, SCAN_AUTO, nullptr, nullptr, bg);
        if (rc) return rc;
        if (prefixed) {          // no occurrence of the prefix anywhere: every boundary is a candidate (gated on best[2])
            rc = launch_scan(p, buf, W, best, s, SCAN_ALL, best + 2, nullptr, bg);
            if (rc) return rc;
        }
    }
    return launch_finish(p, buf, W, best, from_to, 1, s, nullptr, nullptr, nullptr, budgeted ? work + 4 : nullptr);
}

template <typename T>
int grow(T*& ptr, size_t& cap, size_t need_bytes) {
    if (need_bytes <= cap && ptr) return FX_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    size_t want = need_bytes + need_bytes / 8 + 256;
    CUDA_TRY(cudaMalloc(&ptr, want));
    cap = want;
    return FX_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

const char* fx_status_message(int status) {
    if (status < 0) return cudaGetErrorString((cudaError_t)(-status));
    return fx::status_message(status);
}

// where a pattern handle's automata come from: the pattern text (fx_compile) or an anchored DFA explored by the host
// (fx_compile_from_dfa); `.in.` handles compile the anchored form of the same source a second time
struct CompileSource {
    const std::string* pattern = nullptr;
    const fx::DfaInput* dfa = nullptr;
    int compile(int op, int cap, fx::Program& out, bool want_span) const {
        return pattern ? fx::compile_program(*pattern, op, cap, out, want_span) : fx::compile_from_dfa(*dfa, op, cap, out, want_span);
    }
};

static int finish_compile(fx_pattern* p, const CompileSource& src, int op, fx_pattern** out) {
    if (p->prog.status == fx::OK && p->prog.nfa_engine) { *out = p; return fx::OK; }     // NFA engine: no tables to derive
    if (p->prog.status == fx::OK && op != FX_OP_REGEX && (int)p->prog.bt.table.size() * 2 > SMEM_TABLE_LIMIT_BYTES &&
        p->prog.bt.nstates * 8 <= 100 * 1024) {
        // a big boolean automaton: keep its ASCII columns apart if the ASCII bytes fall into at most 4 classes (K1c)
        const fx::ByteTable& bt = p->prog.bt;
        int cols[4] = {-1, -1, -1, -1}, ncols = 0;
        bool ok = true;
        memset(p->cmap4, 0, 256);
        for (int b = 0; b < 128 && ok; b++) {
            const int c = bt.classmap[b];
            int k = 0;
            while (k < ncols && cols[k] != c) k++;
            if (k == ncols) { if (ncols == 4) { ok = false; break; } cols[ncols++] = c; }
            p->cmap4[b] = (uint8_t)k;
        }
        if (ok) {
            p->ctab4.assign((size_t)bt.nstates * 4, 0);
            for (int st = 0; st < bt.nstates; st++)
                for (int k = 0; k < ncols; k++) p->ctab4[(size_t)st * 4 + (size_t)k] = bt.table[((size_t)st << bt.row_shift) + (size_t)cols[k]];
            p->compact = true;
        }
    }
    if (p->prog.status == fx::OK && op == FX_OP_IN && !p->prog.literal_only) {
        // `.in.` consults the prefix prefilter: keep the anchored automaton to replay it exactly when needed.  The same
        // automaton drives the sparse-start kernel; without a prefix it is optional and built under a smaller cap.
        const bool needed = p->prog.prefix_active;
        src.compile(FX_OP_REGEX, needed ? STATE_CAP : SPARSE_STATE_CAP, p->anchored, false);
        if (p->anchored.status == fx::OK) {
            p->has_anchored = true;
            if (needed) p->prefix_mode = prefilter_is_neutral(p->anchored) ? 1 : 2;
            p->sparse = p->prefix_mode != 2 && sparse_first_set(p->anchored.bt, p->first, true);
        } else if (needed) {
            p->prog.status = p->anchored.status;
        }
    }
    if (p->prog.status == fx::OK && op == FX_OP_REGEX && p->prog.has_span_tables) {
        // state-map scan tables: the live states reachable from the start, and the image of all of them under each byte
        const fx::ByteTable& st = p->prog.span_bt;
        std::vector<char> seen((size_t)st.nstates, 0);
        std::vector<int> work{st.start};
        seen[(size_t)st.start] = 1;
        while (!work.empty()) {
            const int u = work.back();
            work.pop_back();
            for (int b = 0; b < 256; b++) {
                const int v = st.direct[(size_t)u * 256 + (size_t)b] & fx::W_SSTATE;
                if (v != 0 && !seen[(size_t)v]) { seen[(size_t)v] = 1; work.push_back(v); }
            }
        }
        for (int u = 1; u < st.nstates; u++) if (seen[(size_t)u]) p->sm_reach.push_back((uint16_t)u);
        p->sm_img.assign(256 * (1 + SM_M), 0);
        for (int b = 0; b < 256; b++) {
            std::vector<int> im;
            for (uint16_t u : p->sm_reach) {
                const int v = st.direct[(size_t)u * 256 + (size_t)b] & fx::W_SSTATE;
                if (v != 0 && std::find(im.begin(), im.end(), v) == im.end()) im.push_back(v);
            }
            p->sm_img[(size_t)b * (1 + SM_M)] = im.size() <= (size_t)SM_M ? (uint16_t)im.size() : (uint16_t)0xFFFF;
            for (size_t k = 0; k < im.size() && k < (size_t)SM_M; k++) p->sm_img[(size_t)b * (1 + SM_M) + 1 + k] = (uint16_t)im[k];
        }
        // synchronising bytes: after c and ANY one more byte at most one live state is left, whatever state read c
        memset(p->sm_sync, 0, 256);
        for (int c = 0; c < 256; c++) {
            const uint16_t n = p->sm_img[(size_t)c * (1 + SM_M)];
            if (n == 0 || n > SM_M) continue;
            bool ok = true;
            for (int d2 = 0; d2 < 256 && ok; d2++) {
                int live = -1;
                for (int k = 0; k < (int)n && ok; k++) {
                    const int u = p->sm_img[(size_t)c * (1 + SM_M) + 1 + (size_t)k];
                    const int v = st.direct[(size_t)u * 256 + (size_t)d2] & fx::W_SSTATE;
                    if (v == 0) continue;
                    if (live >= 0 && live != v) ok = false;
                    live = v;
                }
            }
            p->sm_sync[c] = ok ? 1 : 0;
        }
        p->statemap = true;
    }
    if (p->prog.status == fx::OK && op == FX_OP_REGEX && !p->prog.literal_only) {
        p->sparse = sparse_first_set(p->prog.bt, p->first, false);      // the long-buffer scan can use the SWAR filter
        if (p->prog.prefix_active) {
            // the long-buffer path takes the prefix literal's occurrences as candidates when "non-overlapping occurrences,
            // left to right" (utility_m.f90:58-117) means "all occurrences" -- the literal has no border -- and no suffix
            // literal cuts the list short; a NUL inside the literal would tangle with the frame
            const std::string& pre = p->prog.lit.prefix;
            bool ok = p->prog.lit.suffix.empty() && !pre.empty() && pre.find('\0') == std::string::npos;
            for (size_t k = 1; k < pre.size() && ok; k++)
                if (pre.compare(0, k, pre, pre.size() - k, k) == 0) ok = false;
            p->prefix_scan = ok;
            // is trying every boundary the same as trying the literal's occurrences, as long as the winner begins with
            // the literal's own bytes?  (then the state-map scan may stand in for a candidate scan that ran out of budget)
            p->prefix_neutral = ok && prefilter_is_neutral(p->prog);
        }
    }
    *out = p;
    return p->prog.status;
}


int fx_compile(const void* pattern, int64_t plen, int op, fx_pattern** out) {
    if (!out || plen < 0 || (plen > 0 && !pattern) || op < FX_OP_MATCH || op > FX_OP_REGEX) return FX_ERR_BAD_ARGUMENT;
    fx_pattern* p = new (std::nothrow) fx_pattern();
    if (!p) return fx::ERR_ALLOCATION;
    std::string pat(static_cast<const char*>(pattern), (size_t)plen);
    CompileSource src;
    src.pattern = &pat;
    src.compile(op, env_int("FX_STATE_CAP", STATE_CAP), p->prog, true);      // (FX_STATE_CAP: tests force the NFA engine with a tiny cap)
    return finish_compile(p, src, op, out);
}

// The Fortran-side route: Forgex's own front end has parsed the pattern, extracted the literals and explored the
// automaton eagerly (fortran/forgex_b200_tables_m.F90: a breadth-first search over automaton%construct,
// src/automaton_m.F90:333); this builds every device table from that anchored code-point DFA.
int fx_compile_from_dfa(int op, const int32_t* cuts, int32_t ncls, const int32_t* delta, int32_t nstates, const uint8_t* accept,
                        int32_t q0, const void* all, int64_t all_len, const void* prefix, int64_t prefix_len,
                        const void* suffix, int64_t suffix_len, fx_pattern** out) {
    if (!out || !cuts || !delta || !accept || op < FX_OP_MATCH || op > FX_OP_REGEX || all_len < 0 || prefix_len < 0 || suffix_len < 0)
        return FX_ERR_BAD_ARGUMENT;
    fx_pattern* p = new (std::nothrow) fx_pattern();
    if (!p) return fx::ERR_ALLOCATION;
    fx::DfaInput in;
    in.cuts = cuts; in.delta = delta; in.accept = accept; in.nstates = nstates; in.ncls = ncls; in.q0 = q0;
    if (all_len) in.all.assign(static_cast<const char*>(all), (size_t)all_len);
    if (prefix_len) in.prefix.assign(static_cast<const char*>(prefix), (size_t)prefix_len);
    if (suffix_len) in.suffix.assign(static_cast<const char*>(suffix), (size_t)suffix_len);
    CompileSource src;
    src.dfa = &in;
    src.compile(op, STATE_CAP, p->prog, true);
    return finish_compile(p, src, op, out);
}

// the anchored code-point DFA of an FX_OP_REGEX handle (tests: it is what the Fortran-side route would hand over):
// scalars = {states, classes, q0}; cuts: classes + 1; delta: states x classes (0 = dead); accept: states
int fx_pattern_cp_automaton(const fx_pattern* p, const int32_t** cuts, const int32_t** delta, const uint8_t** accept, int32_t scalars[4]) {
    if (!p || p->prog.status != fx::OK || p->prog.op != FX_OP_REGEX) return FX_ERR_BAD_ARGUMENT;
    const fx::CpAutomaton& a = p->prog.cp;
    static_assert(sizeof(int) == sizeof(int32_t), "int32 views");
    if (cuts) *cuts = reinterpret_cast<const int32_t*>(a.cuts.data());
    if (delta) *delta = reinterpret_cast<const int32_t*>(a.delta.data());
    if (accept) *accept = a.accept.data();
    if (scalars) { scalars[0] = a.nstates; scalars[1] = a.nclasses; scalars[2] = a.q0; scalars[3] = a.start_nul; }
    return FX_OK;
}

// the NFA engine's tables (tests / tools): scalars = {NFA states, 64-bit words per set, classes, exit state, q0 accepting}
int fx_pattern_nfa_tables(const fx_pattern* p, const uint64_t** trans, const uint64_t** q0, const int32_t** cuts, int32_t scalars[5]) {
    if (!p || p->prog.status != fx::OK) return FX_ERR_BAD_ARGUMENT;
    if (!p->prog.nfa_engine) return 1;
    const fx::NfaTables& t = p->prog.nfa_tables;
    if (trans) *trans = t.trans.data();
    if (q0) *q0 = t.q0.data();
    if (cuts) *cuts = reinterpret_cast<const int32_t*>(t.cuts.data());
    if (scalars) { scalars[0] = t.nstates; scalars[1] = t.words; scalars[2] = t.nclasses; scalars[3] = t.exit; scalars[4] = t.q0_accepting ? 1 : 0; }
    return FX_OK;
}

// value-returning / subroutine-shaped forms of the one-pattern-one-text entry points, for `pure` Fortran callers: a
// pure FUNCTION may only have intent(in) / value arguments, so `.in.` and `.match.` come back as the function value
// (1 / 0, or -status on failure), and regex as a procedure without a result (a pure SUBROUTINE may have intent(out)).
int fx_in_value(const void* pattern, int64_t plen, const void* text, int64_t tlen) {
    int r = 0;
    const int rc = fx_in(pattern, plen, text, tlen, &r);
    return rc ? (rc > 0 ? -rc : rc) : r;
}
int fx_match_value(const void* pattern, int64_t plen, const void* text, int64_t tlen) {
    int r = 0;
    const int rc = fx_match(pattern, plen, text, tlen, &r);
    return rc ? (rc > 0 ? -rc : rc) : r;
}
void fx_regex_sub(const void* pattern, int64_t plen, const void* text, int64_t tlen, int64_t* from, int64_t* to, int64_t* length,
                  int* status, int* rc) {
    const int r = fx_regex(pattern, plen, text, tlen, from, to, length, status);
    if (rc) *rc = r;
}

int fx_pattern_free(fx_pattern* p) {
    if (!p) return FX_OK;
    DeviceTables& d = p->dev;
    if (p->dev_touched) {             // also after an upload that failed half-way (every pointer is null or live)
        cudaFree(d.table); cudaFree(d.direct); cudaFree(d.table8); cudaFree(d.classmap); cudaFree(d.flags); cudaFree(d.lits);
        cudaFree(d.a_table); cudaFree(d.a_classmap); cudaFree(d.a_flags);
        cudaFree(d.sp_table); cudaFree(d.sp_direct); cudaFree(d.sp_classmap); cudaFree(d.sp_endinfo);
        cudaFree(d.r_delta); cudaFree(d.r_cuts); cudaFree(d.r_page); cudaFree(d.r_mixed);
        cudaFree(d.sm_reach); cudaFree(d.sm_img); cudaFree(d.sm_sync); cudaFree(d.w_work);
        cudaFree(d.nfa_trans); cudaFree(d.nfa_q0); cudaFree(d.nfa_cuts); cudaFree(d.ctab4); cudaFree(d.cmap4);
        cudaFree(d.w_buf); cudaFree(d.w_off); cudaFree(d.w_out); cudaFree(d.w_span); cudaFree(d.w_best);
    }
    delete p;
    return FX_OK;
}

int fx_pattern_get_info(const fx_pattern* p, fx_pattern_info* info) {
    if (!p || !info) return FX_ERR_BAD_ARGUMENT;
    const fx::Program& g = p->prog;
    memset(info, 0, sizeof(*info));
    info->op = g.op;
    info->status = g.status;
    info->nfa_states = g.nfa_states;
    info->cp_states = g.cp.nstates;
    info->cp_classes = g.cp.nclasses;
    info->byte_states = g.bt.nstates;
    info->byte_classes = g.bt.nclasses;
    info->row_shift = g.bt.row_shift;
    info->table_bytes = (int32_t)g.bt.table.size() * 2;
    info->direct_bytes = (int32_t)g.bt.direct.size() * 2;
    info->literal_all_len = (int32_t)g.lit.all.size();
    info->literal_prefix_len = (int32_t)g.lit.prefix.size();
    info->literal_suffix_len = (int32_t)g.lit.suffix.size();
    info->literal_only = g.literal_only ? 1 : 0;
    info->residency = p->last_residency;
    info->direct = p->last_direct;
    info->prefix_mode = p->prefix_mode;
    info->sparse = p->sparse ? 1 : 0;
    info->sparse_ranges = p->sparse ? p->first.nr : 0;
    info->sparse_high = p->sparse && p->first.high ? 1 : 0;
    info->sparse_second = p->sparse && p->first.two ? p->first.second : -1;
    for (int r = 0; r < 4; r++) {
        info->sparse_lo[r] = p->sparse && r < p->first.nr ? p->first.lo[r] : 0;
        info->sparse_hi[r] = p->sparse && r < p->first.nr ? p->first.hi[r] : 0;
    }
    info->sparse_used = p->last_sparse;
    info->prefix_scan = p->prefix_scan ? 1 : 0;
    info->nfa_engine = g.nfa_engine ? 1 : 0;
    info->compact_used = p->last_compact;
    info->statemap = p->statemap ? 1 : 0;
    info->statemap_used = p->last_statemap;
    info->gated = g.op == FX_OP_REGEX || g.nfa_engine ? 0 : gated_mode(p, g.op);
    return FX_OK;
}

int fx_pattern_set_residency(fx_pattern* p, int residency) {
    if (!p || residency < FX_TABLE_AUTO || residency > FX_TABLE_GLOBAL) return FX_ERR_BAD_ARGUMENT;
    p->residency = residency;
    return FX_OK;
}

int fx_pattern_literals(const fx_pattern* p, void* all, void* prefix, void* suffix) {
    if (!p) return FX_ERR_BAD_ARGUMENT;
    const fx::Literals& L = p->prog.lit;
    if (all && !L.all.empty()) memcpy(all, L.all.data(), L.all.size());
    if (prefix && !L.prefix.empty()) memcpy(prefix, L.prefix.data(), L.prefix.size());
    if (suffix && !L.suffix.empty()) memcpy(suffix, L.suffix.data(), L.suffix.size());
    return FX_OK;
}

int fx_pattern_tables(const fx_pattern* p, const uint16_t** table, const uint16_t** direct, const uint8_t** classmap,
                      const uint8_t** flags, int32_t scalars[6]) {
    if (!p || p->prog.status != fx::OK) return FX_ERR_BAD_ARGUMENT;
    const fx::ByteTable& bt = p->prog.bt;
    if (table) *table = bt.table.data();
    if (direct) *direct = bt.direct.data();
    if (classmap) *classmap = bt.classmap;
    if (flags) *flags = bt.flags.data();
    if (scalars) {
        scalars[0] = bt.start; scalars[1] = bt.start_nul; scalars[2] = bt.q0; scalars[3] = bt.matched;
        scalars[4] = bt.q0_accepting ? 1 : 0;
        scalars[5] = bt.result_threshold;
    }
    return FX_OK;
}

int fx_pattern_span_tables(const fx_pattern* p, const uint16_t** direct, const uint8_t** endinfo, int32_t scalars[4],
                           const uint16_t** rdelta, const uint8_t** rpage, const uint8_t** rmixed, const int32_t** cuts,
                           int32_t rscalars[4]) {
    if (!p || p->prog.status != fx::OK) return FX_ERR_BAD_ARGUMENT;
    if (!p->prog.has_span) return 1;      // the pattern has no linear-time span path
    const fx::ByteTable& st = p->prog.span_bt;
    const fx::RevAutomaton& rv = p->prog.rev;
    if (direct) *direct = st.direct.data();
    if (endinfo) *endinfo = st.endinfo.data();
    if (scalars) { scalars[0] = st.nstates; scalars[1] = st.start; scalars[2] = (st.flags[(size_t)st.start] & fxk::SF_ACC) ? 1 : 0; scalars[3] = 0; }
    if (rdelta) *rdelta = rv.delta16.data();
    if (rpage) *rpage = rv.page.empty() ? nullptr : rv.page.data();
    if (rmixed) *rmixed = rv.mixed.empty() ? nullptr : rv.mixed.data();
    static_assert(sizeof(int) == sizeof(int32_t), "cuts are exposed as int32");
    if (cuts) *cuts = reinterpret_cast<const int32_t*>(rv.cuts.data());
    if (rscalars) { rscalars[0] = rv.nstates; rscalars[1] = rv.nclasses; rscalars[2] = rv.start; rscalars[3] = (int32_t)(rv.mixed.size() / 64); }
    return FX_OK;
}

int fx_is_valid_regex(const void* pattern, int64_t plen, int* status) {  // forgex.F90:58-71
    if (plen < 0 || (plen > 0 && !pattern)) return FX_ERR_BAD_ARGUMENT;
    fx::Syntax syn;
    fx::parse_pattern(fx::prepare_pattern(std::string(static_cast<const char*>(pattern), (size_t)plen), false), syn);
    if (status) *status = syn.status;
    return syn.valid() ? 1 : 0;
}

// is_valid_regex is `pure elemental` in the reference (forgex.F90:58-71): over an array of patterns it answers per
// element.  Batch form: patterns as a flat buffer + n+1 ascending offsets; valid[i] = 1/0, status[i] = SYNTAX_* code
// (error_m.F90:12-38).  Host-only, like the reference's (pattern parsing is not part of the matching loop).
int fx_is_valid_regex_batch(const void* patterns, const int64_t* offsets, int64_t n, uint8_t* valid, int32_t* status) {
    if (n < 0 || (n > 0 && (!offsets || (!valid && !status)))) return FX_ERR_BAD_ARGUMENT;
    const char* base = static_cast<const char*>(patterns);
    for (int64_t i = 0; i < n; i++) {
        const int64_t a = offsets[i], b = offsets[i + 1];
        if (a < 0 || b < a || (b > a && !base)) return FX_ERR_BAD_ARGUMENT;
        fx::Syntax syn;
        fx::parse_pattern(fx::prepare_pattern(std::string(base ? base + a : "", (size_t)(b - a)), false), syn);
        if (valid) valid[i] = syn.valid() ? 1 : 0;
        if (status) status[i] = syn.status;
    }
    return FX_OK;
}

// ---- device-pointer entry points ------------------------------------------------------------
int fx_match_fixed_dev(fx_pattern* p, const uint8_t* d_buf, int64_t n, int64_t stride, uint8_t* d_out, void* stream) {
    int rc = check_ready(p, FX_OP_MATCH);
    if (rc) return rc;
    return launch_fixed<0>(p, d_buf, n, stride, d_out, (cudaStream_t)stream);
}
int fx_in_fixed_dev(fx_pattern* p, const uint8_t* d_buf, int64_t n, int64_t stride, uint8_t* d_out, void* stream) {
    int rc = check_ready(p, FX_OP_IN);
    if (rc) return rc;
    return launch_fixed<1>(p, d_buf, n, stride, d_out, (cudaStream_t)stream);
}
int fx_match_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                       uint8_t* d_out, void* stream) {
    int rc = check_ready(p, FX_OP_MATCH);
    if (rc) return rc;
    return launch_ragged<0>(p, d_buf, d_offsets, n, total_bytes, d_out, (cudaStream_t)stream);
}
int fx_in_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                    uint8_t* d_out, void* stream) {
    int rc = check_ready(p, FX_OP_IN);
    if (rc) return rc;
    return launch_ragged<1>(p, d_buf, d_offsets, n, total_bytes, d_out, (cudaStream_t)stream);
}
int fx_regex_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                       int64_t* d_from, int64_t* d_to, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    return launch_regex_ragged(p, d_buf, d_offsets, n, total_bytes, d_from, d_to, (cudaStream_t)stream);
}
int64_t fx_regex_buffer_work_bytes(int64_t len) { return (int64_t)buffer_work_bytes(len); }
int fx_regex_buffer_dev(fx_pattern* p, const uint8_t* d_buf, int64_t len, int64_t* d_from_to, void* d_work, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (!d_work) return FX_ERR_BAD_ARGUMENT;
    return launch_buffer(p, d_buf, len, d_from_to, static_cast<unsigned long long*>(d_work), (cudaStream_t)stream);
}

int fx_buffer_scan_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t start_lo, int64_t start_hi,
                       int64_t origin, int is_first, int is_last, uint64_t* d_best, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (!d_best) return FX_ERR_BAD_ARGUMENT;
    ScanWindow W{window_len, start_lo, start_hi, origin, is_first ? 1 : 0, is_last ? 1 : 0};
    return launch_scan(p, d_window, W, reinterpret_cast<unsigned long long*>(d_best), (cudaStream_t)stream, SCAN_AUTO);
}
int fx_buffer_scan_all_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t start_lo, int64_t start_hi,
                           int64_t origin, int is_first, int is_last, uint64_t* d_best, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (!d_best) return FX_ERR_BAD_ARGUMENT;
    ScanWindow W{window_len, start_lo, start_hi, origin, is_first ? 1 : 0, is_last ? 1 : 0};
    return launch_scan(p, d_window, W, reinterpret_cast<unsigned long long*>(d_best), (cudaStream_t)stream, SCAN_ALL);
}
int fx_buffer_finish_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t origin, int is_last,
                         const uint64_t* d_key, int64_t* d_from_to, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (!d_key || !d_from_to) return FX_ERR_BAD_ARGUMENT;
    ScanWindow W{window_len, 0, window_len, origin, origin == 0 ? 1 : 0, is_last ? 1 : 0};
    return launch_finish(p, d_window, W, reinterpret_cast<const unsigned long long*>(d_key), d_from_to, 0, (cudaStream_t)stream);
}

// ---- linear-time window form: slab maps of the state-map scan, their combine, the backward walk across windows ----
static_assert(FX_STATEMAP_MAP_WORDS == 2 + 3 * 32 && FX_STATEMAP_UNKNOWN == SM_MAP_UNKNOWN, "slab map layout");
static_assert(FX_STATEMAP_WALK_NEW == SM_WALK_NEW && FX_STATEMAP_WALK_DONE == SM_WALK_DONE, "walk layout");

// which patterns the window form serves (host-only: no device needed)
static int statemap_window_served(const fx_pattern* p) {
    if (!p) return FX_ERR_BAD_ARGUMENT;
    if (p->prog.status != fx::OK) return p->prog.status;
    if (p->prog.op != FX_OP_REGEX) return FX_ERR_BAD_ARGUMENT;
    if (p->prog.nfa_engine) return FX_ERR_DFA_STATE_CAP;
    // a prefix literal restricts Forgex's candidates to its occurrences, which may lie in another slab
    if (p->prog.literal_only || p->prog.prefix_active) return FX_ERR_PREFILTER_UNSUPPORTED;
    if (!p->statemap) return FX_ERR_DFA_STATE_CAP;
    return FX_OK;
}

int fx_statemap_window_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t slab_lo, int64_t slab_hi,
                           int64_t origin, int64_t* d_map, void* d_work, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if ((rc = statemap_window_served(p))) return rc;
    if (!d_map || !d_work || (!d_window && window_len > 0) || origin < 0 || slab_lo < 0 || slab_lo > slab_hi ||
        slab_hi > window_len)
        return FX_ERR_BAD_ARGUMENT;
    const int64_t back = origin + slab_lo < SM_LOOKBACK ? origin + slab_lo : SM_LOOKBACK;
    if (slab_lo < back) return FX_ERR_BAD_ARGUMENT;          // the look-back in front of the slab is missing
    SpanParams sp;
    fill_span_params(p, sp);
    return launch_statemap_scan(p, sp, d_window + slab_lo, slab_hi - slab_lo, back, origin + slab_lo,
                                static_cast<unsigned long long*>(d_work), reinterpret_cast<long long*>(d_map),
                                (cudaStream_t)stream, nullptr, true);
}

int fx_statemap_combine(const fx_pattern* p, const int64_t* maps, int64_t nmaps, int64_t text_len, int64_t out[2]) {
    int rc = statemap_window_served(p);
    if (rc) return rc;
    if (!out || nmaps < 0 || (nmaps > 0 && !maps) || text_len < 0) return FX_ERR_BAD_ARGUMENT;
    const fx::ByteTable& st = p->prog.span_bt;
    int64_t s = st.start;
    int64_t last = (st.flags[(size_t)st.start] & fxk::SF_ACC) ? 0 : -1;
    out[0] = -1; out[1] = 0;
    for (int64_t i = 0; i < nmaps && s != 0; i++) {
        const int64_t* m = maps + i * FX_STATEMAP_MAP_WORDS;
        if (m[0] == 2) continue;                             // empty slab: the identity
        if (m[0] != 0 || m[1] < 0 || m[1] > 32) { out[1] = 1; return FX_OK; }
        int hit = -1;
        for (int k = 0; k < (int)m[1]; k++) if (m[2 + k] == s) hit = k;
        if (hit < 0 || m[66 + hit] == FX_STATEMAP_UNKNOWN) { out[1] = 1; return FX_OK; }
        s = m[34 + hit];
        if (s < 0 || s >= st.nstates) return FX_ERR_BAD_ARGUMENT;
        if (m[66 + hit] >= 0) last = m[66 + hit];
    }
    if (s != 0) {                                            // end of the text: pending bytes replay, the trailing NUL is consumed
        const uint32_t e = st.endinfo[(size_t)s];
        if (e & 3u) last = text_len + 1 - (int64_t)(e & 3u);
        if (e & 4u) last = text_len + 1;
    }
    out[0] = last;
    return FX_OK;
}

int fx_statemap_back_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t origin, int64_t text_len,
                         int64_t* d_walk, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if ((rc = statemap_window_served(p))) return rc;
    if (!d_walk || (!d_window && window_len > 0) || window_len < 0 || origin < 0 || origin + window_len > text_len)
        return FX_ERR_BAD_ARGUMENT;
    SpanParams sp;
    fill_span_params(p, sp);
    k_statemap_back<<<1, 1, 0, (cudaStream_t)stream>>>(sp, d_window, origin, window_len, text_len, reinterpret_cast<long long*>(d_walk));
    g_launches++;
    return cuda_status(cudaGetLastError());
}

// ---- all matches / match counts (the loop a caller of regex() writes: match, then regex() again on text(to+1:)) ----
int fx_regex_count_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                             int64_t* d_counts, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (n < 0 || total_bytes < 0 || !d_counts) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    if (p->prog.nfa_engine) return FX_ERR_DFA_STATE_CAP;        // (counting needs the table engine)
    Plan pl;
    if ((rc = make_plan(p, pl))) return rc;
    SpanParams sp;
    memset(&sp, 0, sizeof(sp));
    long long want = (n + 255) / 256, cap = (long long)p->dev.sm_count * 16;
    const int grid = (int)(want < cap ? want : cap);
    if (p->prog.has_span && env_int("FX_SPAN_LINEAR", 1)) {
        fill_span_params(p, sp);
        k_regex_count<true><<<grid, 256, 0, (cudaStream_t)stream>>>(pl.kp, sp, d_buf, d_offsets, n, d_counts);
    } else {
        k_regex_count<false><<<grid, 256, 0, (cudaStream_t)stream>>>(pl.kp, sp, d_buf, d_offsets, n, d_counts);
    }
    g_launches++;
    return cuda_status(cudaGetLastError());
}

// One buffer: every match, in order.  d_from / d_to receive the first `capacity` spans (64-bit, 1-based inclusive, in
// coordinates of the whole buffer); *count (host) = the number of matches, which may exceed capacity.  The search for
// the next match is the long-buffer search on the rest; short hops are taken on the device, a thousand per launch.
// Synchronises `stream` (once per far match / per thousand near ones).
int fx_regex_buffer_all_dev(fx_pattern* p, const uint8_t* d_buf, int64_t len, int64_t* d_from, int64_t* d_to, int64_t capacity,
                            int64_t* count, void* d_work, void* stream) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (len < 0 || capacity < 0 || !count || !d_work || (capacity > 0 && (!d_from || !d_to))) return FX_ERR_BAD_ARGUMENT;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long* work = static_cast<unsigned long long*>(d_work);
    // the loop's own state sits behind the scans' flags in the work area (see WORK_HEAD): words [24..28] state, of which
    // [28] is the work-budget flag, and [30..31] from_to of a far step.  The two must not overlap: a far match's `from`
    // in the budget word would turn a loop that then ends in the local step into FX_ERR_WORK_BUDGET.
    int64_t* state = reinterpret_cast<int64_t*>(work + 24);
    int64_t* ft = reinterpret_cast<int64_t*>(work + 30);
    if (p->prog.nfa_engine) return FX_ERR_DFA_STATE_CAP;
    CUDA_TRY(cudaMemsetAsync(state, 0, 8 * 8, s));
    Plan pl;
    if ((rc = make_plan(p, pl))) return rc;
    SpanParams sp;
    memset(&sp, 0, sizeof(sp));
    const bool local = p->prog.has_span && env_int("FX_ALL_LOCAL", 1);
    if (local) fill_span_params(p, sp);
    int64_t host_state[5] = {0, 0, 0, 0, 0};
    for (;;) {
        if (local) {
            k_buffer_all_local<<<1, 1, 0, s>>>(pl.kp, sp, d_buf, len, state, d_from, d_to, capacity, 1024, (int64_t)env_int("FX_ALL_REACH", 1 << 16));
            g_launches++;
            CUDA_TRY(cudaMemcpyAsync(host_state, state, 40, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaStreamSynchronize(s));
            if (host_state[2]) break;
            if (!host_state[3]) continue;                   // a thousand near matches taken: go on
        }
        const int64_t pos = host_state[0];
        if ((rc = launch_buffer(p, d_buf + pos, len - pos, ft, work, s))) return rc;
        k_buffer_all_take<<<1, 1, 0, s>>>(ft, state, d_from, d_to, capacity);
        g_launches++;
        CUDA_TRY(cudaMemcpyAsync(host_state, state, 40, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        if (host_state[2]) break;
    }
    *count = host_state[1];
    if (host_state[4]) return FX_ERR_WORK_BUDGET;
    return FX_OK;
}

// ---- host-pointer entry points ----------------------------------------------------------------
static int host_bool_fixed(fx_pattern* p, int op, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out) {
    int rc = check_ready(p, op);
    if (rc) return rc;
    if (n < 0 || stride < 0) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    std::lock_guard<std::mutex> lock(p->mu);
    DeviceTables& d = p->dev;
    if (stride > 0 && n > (int64_t)((~(size_t)0 >> 2) / (size_t)stride)) return FX_ERR_BAD_ARGUMENT;   // n * stride overflows
    size_t bytes = (size_t)n * (size_t)stride;
    if ((rc = grow(d.w_buf, d.w_buf_cap, bytes + 64))) return rc;
    if ((rc = grow(d.w_out, d.w_out_cap, (size_t)n))) return rc;
    if (bytes) CUDA_TRY(cudaMemcpyAsync(d.w_buf, buf, bytes, cudaMemcpyHostToDevice, 0));
    rc = op == FX_OP_MATCH ? launch_fixed<0>(p, d.w_buf, n, stride, d.w_out, 0) : launch_fixed<1>(p, d.w_buf, n, stride, d.w_out, 0);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, d.w_out, (size_t)n, cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    return FX_OK;
}
int fx_match_fixed(fx_pattern* p, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out) {
    return host_bool_fixed(p, FX_OP_MATCH, buf, n, stride, out);
}
int fx_in_fixed(fx_pattern* p, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out) {
    return host_bool_fixed(p, FX_OP_IN, buf, n, stride, out);
}

static int host_stage_ragged(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, int64_t& total) {
    DeviceTables& d = p->dev;
    int64_t base = offsets[0];
    total = offsets[n] - base;
    if (total < 0 || base != 0) return FX_ERR_BAD_ARGUMENT;   // offsets must start at 0
    int rc;
    if ((rc = grow(d.w_buf, d.w_buf_cap, (size_t)total + 64))) return rc;
    if ((rc = grow(d.w_off, d.w_off_cap, (size_t)(n + 1) * 8))) return rc;
    // offsets first: they are checked on the device (ascending, inside [0, total]) while the text is still on its way
    CUDA_TRY(cudaMemcpyAsync(d.w_off, offsets, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, 0));
    int* d_bad = reinterpret_cast<int*>(d.w_best + 3);
    CUDA_TRY(cudaMemsetAsync(d_bad, 0, 4, 0));
    {
        long long want = (n + 255) / 256, cap = (long long)d.sm_count * 8;
        k_check_offsets<<<(int)(want < cap ? want : cap), 256, 0, 0>>>(d.w_off, n, total, d_bad);
        g_launches++;
    }
    int bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, 0));
    if (total) CUDA_TRY(cudaMemcpyAsync(d.w_buf, buf, (size_t)total, cudaMemcpyHostToDevice, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    if (bad) return FX_ERR_BAD_ARGUMENT;      // no kernel has touched the text through these offsets
    return FX_OK;
}
static int host_bool_ragged(fx_pattern* p, int op, const uint8_t* buf, const int64_t* offsets, int64_t n, uint8_t* out) {
    int rc = check_ready(p, op);
    if (rc) return rc;
    if (n < 0 || !offsets) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    std::lock_guard<std::mutex> lock(p->mu);
    DeviceTables& d = p->dev;
    int64_t total = 0;
    if ((rc = host_stage_ragged(p, buf, offsets, n, total))) return rc;
    if ((rc = grow(d.w_out, d.w_out_cap, (size_t)n))) return rc;
    rc = op == FX_OP_MATCH ? launch_ragged<0>(p, d.w_buf, d.w_off, n, total, d.w_out, 0)
                           : launch_ragged<1>(p, d.w_buf, d.w_off, n, total, d.w_out, 0);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, d.w_out, (size_t)n, cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    return FX_OK;
}
int fx_match_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, uint8_t* out) {
    return host_bool_ragged(p, FX_OP_MATCH, buf, offsets, n, out);
}
int fx_in_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, uint8_t* out) {
    return host_bool_ragged(p, FX_OP_IN, buf, offsets, n, out);
}
int fx_regex_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, int64_t* from, int64_t* to) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (n < 0 || !offsets) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    std::lock_guard<std::mutex> lock(p->mu);
    DeviceTables& d = p->dev;
    int64_t total = 0;
    if ((rc = host_stage_ragged(p, buf, offsets, n, total))) return rc;
    if ((rc = grow(d.w_span, d.w_span_cap, (size_t)n * 16))) return rc;
    rc = launch_regex_ragged(p, d.w_buf, d.w_off, n, total, d.w_span, d.w_span + n, 0);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(from, d.w_span, (size_t)n * 8, cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaMemcpyAsync(to, d.w_span + n, (size_t)n * 8, cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    return FX_OK;
}
int fx_regex_count_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, int64_t* counts) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (n < 0 || !offsets || !counts) return FX_ERR_BAD_ARGUMENT;
    if (n == 0) return FX_OK;
    std::lock_guard<std::mutex> lock(p->mu);
    DeviceTables& d = p->dev;
    int64_t total = 0;
    if ((rc = host_stage_ragged(p, buf, offsets, n, total))) return rc;
    if ((rc = grow(d.w_span, d.w_span_cap, (size_t)n * 8))) return rc;
    if ((rc = fx_regex_count_batch_dev(p, d.w_buf, d.w_off, n, total, d.w_span, nullptr))) return rc;
    CUDA_TRY(cudaMemcpyAsync(counts, d.w_span, (size_t)n * 8, cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    return FX_OK;
}
int fx_regex_buffer_all(fx_pattern* p, const uint8_t* buf, int64_t len, int64_t* from, int64_t* to, int64_t capacity, int64_t* count) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (len < 0 || capacity < 0 || !count) return FX_ERR_BAD_ARGUMENT;
    std::lock_guard<std::mutex> lock(p->mu);
    DeviceTables& d = p->dev;
    if ((rc = grow(d.w_buf, d.w_buf_cap, (size_t)len + 64))) return rc;
    if ((rc = grow(d.w_span, d.w_span_cap, (size_t)capacity * 16 + 16))) return rc;
    if ((rc = grow(d.w_work, d.w_work_cap, buffer_work_bytes(len)))) return rc;
    if (len) CUDA_TRY(cudaMemcpyAsync(d.w_buf, buf, (size_t)len, cudaMemcpyHostToDevice, 0));
    if ((rc = fx_regex_buffer_all_dev(p, d.w_buf, len, d.w_span, d.w_span + capacity, capacity, count, d.w_work, nullptr))) return rc;
    const int64_t k = *count < capacity ? *count : capacity;
    if (k > 0) {
        CUDA_TRY(cudaMemcpyAsync(from, d.w_span, (size_t)k * 8, cudaMemcpyDeviceToHost, 0));
        CUDA_TRY(cudaMemcpyAsync(to, d.w_span + capacity, (size_t)k * 8, cudaMemcpyDeviceToHost, 0));
        CUDA_TRY(cudaStreamSynchronize(0));
    }
    return FX_OK;
}
int fx_regex_buffer(fx_pattern* p, const uint8_t* buf, int64_t len, int64_t* from, int64_t* to) {
    int rc = check_ready(p, FX_OP_REGEX);
    if (rc) return rc;
    if (len < 0) return FX_ERR_BAD_ARGUMENT;
    std::lock_guard<std::mutex> lock(p->mu);
    DeviceTables& d = p->dev;
    if ((rc = grow(d.w_buf, d.w_buf_cap, (size_t)len + 64))) return rc;
    if ((rc = grow(d.w_span, d.w_span_cap, 16))) return rc;
    if ((rc = grow(d.w_work, d.w_work_cap, buffer_work_bytes(len)))) return rc;
    if (len) CUDA_TRY(cudaMemcpyAsync(d.w_buf, buf, (size_t)len, cudaMemcpyHostToDevice, 0));
    rc = launch_buffer(p, d.w_buf, len, d.w_span, reinterpret_cast<unsigned long long*>(d.w_work), 0);
    if (rc) return rc;
    int64_t ft[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(ft, d.w_span, 16, cudaMemcpyDeviceToHost, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    if (ft[0] == -2 && ft[1] == -2) return FX_ERR_WORK_BUDGET;
    if (from) *from = ft[0];
    if (to) *to = ft[1];
    return FX_OK;
}

// ---- one pattern, one text ----------------------------------------------------------------------
int fx_in(const void* pattern, int64_t plen, const void* text, int64_t tlen, int* result) {
    if (!result || tlen < 0) return FX_ERR_BAD_ARGUMENT;
    fx_pattern* p = nullptr;
    int rc = fx_compile(pattern, plen, FX_OP_IN, &p);
    if (rc >= 1 && rc <= 24) { *result = 0; fx_pattern_free(p); return FX_OK; }   // invalid pattern -> .false. (forgex.F90:101-104)
    if (rc) { fx_pattern_free(p); return rc; }
    uint8_t out = 0;
    rc = fx_in_fixed(p, static_cast<const uint8_t*>(text), 1, tlen, &out);
    *result = out;
    fx_pattern_free(p);
    return rc;
}
int fx_match(const void* pattern, int64_t plen, const void* text, int64_t tlen, int* result) {
    if (!result || tlen < 0) return FX_ERR_BAD_ARGUMENT;
    fx_pattern* p = nullptr;
    int rc = fx_compile(pattern, plen, FX_OP_MATCH, &p);
    if (rc >= 1 && rc <= 24) { *result = 0; fx_pattern_free(p); return FX_OK; }   // forgex.F90:197-200
    if (rc) { fx_pattern_free(p); return rc; }
    uint8_t out = 0;
    rc = fx_match_fixed(p, static_cast<const uint8_t*>(text), 1, tlen, &out);
    *result = out;
    fx_pattern_free(p);
    return rc;
}
int fx_regex(const void* pattern, int64_t plen, const void* text, int64_t tlen, int64_t* from, int64_t* to,
             int64_t* length, int* status) {
    if (tlen < 0) return FX_ERR_BAD_ARGUMENT;
    fx_pattern* p = nullptr;
    int rc = fx_compile(pattern, plen, FX_OP_REGEX, &p);
    if (status) *status = (rc >= 1 && rc <= 24) ? rc : 0;
    if (rc >= 1 && rc <= 24) {   // forgex.F90:266-274
        if (from) *from = -9999;
        if (to) *to = -9999;
        if (length) *length = 0;
        fx_pattern_free(p);
        return FX_OK;
    }
    if (rc) { fx_pattern_free(p); return rc; }
    int64_t off[2] = {0, tlen}, f = 0, t = 0;
    rc = fx_regex_batch(p, static_cast<const uint8_t*>(text), off, 1, &f, &t);
    if (from) *from = f;
    if (to) *to = t;
    if (length) *length = (f > 0 && t > 0) ? t - f + 1 : 0;
    fx_pattern_free(p);
    return rc;
}

int64_t fx_launch_count(void) { return g_launches.load(); }

}  // extern "C"
