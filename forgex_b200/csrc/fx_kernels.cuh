// fx_kernels.cuh -- sm_100a kernels of the Forgex matching path.
//
// Every kernel is "walk the byte-level DFA table, read a flag": the transition loop that the
// reference executes per character in do_matching_exactly / do_matching_including
// (/root/reference/src/api_internal_m.F90:119-137, :258-295) with automaton%construct
// (/root/reference/src/automaton_m.F90:333-381) replaced by one table lookup per BYTE.
// This is HBM-bound integer work: no tensor cores.  What matters (DESIGN.md): text is read
// from HBM exactly once in coalesced 16-byte pieces (TMA bulk copies into shared memory for
// ragged batches), the table lives in shared memory, one dependent LDS per byte per thread and
// enough threads per SM to hide its latency.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fxk {

// word layout (must match fx_internal.hpp)
static constexpr uint32_t W_ACC = 0x8000u, W_INTER = 0x4000u, W_STATE = 0x3FFFu;
static constexpr uint32_t SF_ACC = 1, SF_END = 2, SF_INTER = 4, SF_MATCHED = 8, SF_FAILACC1 = 16;

struct KParams {
    const uint16_t* table;    // selected table in global memory (class-compressed or 256-column)
    const uint8_t* classmap;  // 256 bytes
    const uint8_t* flags;     // nstates bytes
    const uint8_t* lits;      // all | prefix | suffix, back to back
    int table_words;
    int nstates;
    int row_shift;            // 8 for the 256-column table
    int start, start_nul, q0, q0_accepting;
    int all_len, pre_len, suf_len;
    int all_active;           // `all` is not blank: literal fast path (forgex.F90:111-130, :207-213, :281-307)
    int pre_active, suf_active;  // prefix / suffix not blank
    // `.in.` with an active prefix: the anchored (REGEX-mode, flag-bit) class-compressed table, used to
    // replay Forgex's prefix-candidate search exactly (api_internal_m.F90:76-164) when it can matter
    const uint16_t* a_table;
    const uint8_t* a_classmap;
    const uint8_t* a_flags;
    int a_row_shift, a_start_nul, a_q0;
    int prefix_mode;          // 0: none; 1: neutral unless the text holds bytes >= 0x80; 2: always replay
    // boolean tables: one-byte entries (<= 255 states) and "state >= result_threshold <=> result is true"
    const uint8_t* table8;
    int result_threshold;
    // the class-compressed table in global memory, whatever `table` points to (slow paths, finish kernel)
    const uint16_t* ctable;
    int c_row_shift;
    long long* steps_left;    // nullptr except in k_buffer_sequential (work budget of the single-thread replay)
};

// ---- small PTX helpers ---------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {  // streaming 16-byte load, no L1 allocation
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
// The sweep load of K4: a plain read-only load that allocates in L1.  Measured on C4
// (profiles/r02_prof_c4_sweep_load_policy.txt): with no L1 allocation (ldg_nc_v4, the K2c choice) the unit phase's
// re-read of a candidate unit, microseconds after the sweep read it, MISSES L2 and goes to DRAM at 64-byte granularity
// -- 3.55 GB of DRAM reads for 2.15 GB of text; this load brings that to 2.34 GB and the search from 3.43 to 3.27 ms
// per 8 GiB.
__device__ __forceinline__ uint4 ldg_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg_nc_v2(const void* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count));
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t phase) {
    uint32_t ok;
    do {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(ok) : "r"(mbar), "r"(phase) : "memory");
    } while (!ok);
}
// TMA 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}

// ---- table access --------------------------------------------------------------------------
// KIND 0: one-byte entries, 256 columns, shared memory (boolean tables with <= 255 states).  A row is 64
//         words: for ASCII text the 32 banks see distinct words, so lanes in the same state never conflict.
// KIND 1: 16-bit entries, 256 columns, shared memory (span tables, flag bits in the word)
// KIND 2: 16-bit entries, class-compressed rows + classmap, shared memory
// KIND 3: 16-bit entries, class-compressed rows + classmap, global memory through L1/L2
// KIND 0 rows are padded to 65 words in shared memory: with 64-word rows the bank of a lookup depends on the byte
// alone, so lanes that sit in DIFFERENT states and read the same byte value (digits, the dead state's row ...) collide.
static constexpr int ROW8 = 260;
template <int KIND>
struct Table {
    uint32_t s_table, s_cmap;  // shared addresses
    const uint16_t* g_table;
    const uint8_t* g_cmap;
    int shift;
    __device__ __forceinline__ uint32_t next(uint32_t state, uint32_t byte) const {
        if (KIND == 0) return lds_u8(s_table + state * ROW8 + byte);
        if (KIND == 1) return lds_u16(s_table + (((state << 8) | byte) << 1));
        if (KIND == 2) return lds_u16(s_table + (((state << shift) + lds_u8(s_cmap + byte)) << 1));
        return __ldg(g_table + ((state << shift) + __ldg(g_cmap + byte)));
    }
};

// cooperative copy of the table into shared memory; returns the filled Table
template <int KIND>
__device__ __forceinline__ Table<KIND> stage_table(const KParams& p, uint8_t* smem_table, uint8_t* smem_cmap) {
    Table<KIND> t;
    t.g_table = p.table; t.g_cmap = p.classmap; t.shift = p.row_shift;
    t.s_table = 0; t.s_cmap = 0;
    if (KIND != 3) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(KIND == 0 ? (const void*)p.table8 : (const void*)p.table);
        uint32_t* dst = reinterpret_cast<uint32_t*>(smem_table);
        const int words32 = KIND == 0 ? p.nstates * 64 : (p.table_words + 1) >> 1;
        if (KIND == 0) for (int i = threadIdx.x; i < words32; i += blockDim.x) dst[(i >> 6) * (ROW8 / 4) + (i & 63)] = __ldg(src + i);
        else for (int i = threadIdx.x; i < words32; i += blockDim.x) dst[i] = __ldg(src + i);
        if (KIND == 2)
            for (int i = threadIdx.x; i < 64; i += blockDim.x)
                reinterpret_cast<uint32_t*>(smem_cmap)[i] = __ldg(reinterpret_cast<const uint32_t*>(p.classmap) + i);
        t.s_table = smem_u32(smem_table);
        t.s_cmap = smem_u32(smem_cmap);
    }
    return t;
}

__device__ __forceinline__ bool result_flag(const KParams& p, uint32_t state) {
    return state >= (uint32_t)p.result_threshold;   // boolean tables number their result states last
}

// Text of length 0, or one blank, never reaches the `.in.`/`regex` loop (api_internal_m.F90:68-74);
// empty text never reaches the `.match.` loop (:247-250).
template <int OP>
__device__ __forceinline__ bool degenerate_text(int64_t len, uint32_t first_byte) {
    if (OP == 0) return len == 0;
    return len == 0 || (len == 1 && first_byte == 0x20);
}

// ---------------------------------------------------------------------------------------------
// spans: leftmost start, longest end -- the loop of do_matching_including (api_internal_m.F90:108-164)
// ---------------------------------------------------------------------------------------------
struct FetchGeneric {
    const uint8_t* s;
    __device__ __forceinline__ uint32_t operator()(int64_t i) const { return s[i]; }
};
struct FetchGlobal {
    const uint8_t* s;
    __device__ __forceinline__ uint32_t operator()(int64_t i) const { return __ldg(s + i); }
};
struct FetchShared {
    uint32_t a;
    __device__ __forceinline__ uint32_t operator()(int64_t i) const { return lds_u8(a + (uint32_t)i); }
};

// the anchored automaton a span search runs on (flag-bit table)
struct Anchored {
    const uint8_t* flags;
    int start_nul, q0;
    long long* steps_left = nullptr;   // single-thread replay over a long buffer: byte steps it may still take (see k_buffer_sequential)
};
static constexpr int64_t OUT_OF_BUDGET = -3;     // an attempt that ran out of steps (never a legal `last`)

// One anchored attempt starting with `st` before text index `pos`.  `last` is -1 or the number of
// text bytes consumed at the last accepting boundary (len+1 = the trailing NUL was consumed too).
// A malformed multi-byte sequence is replayed by the table as U+FFFF per byte; accepts that fall
// between those replayed bytes are recovered from the SF_FAILACC bits of the in-sequence state.
template <class TBL, class FETCH>
__device__ __forceinline__ int64_t run_attempt(const Anchored& A, const TBL& T, FETCH fetch, int64_t len, uint32_t st,
                                               int64_t pos, int64_t last) {
    uint32_t w = st;           // previous word (INTER bit tells whether we are inside a sequence)
    int64_t seq = 0;           // index of the lead byte of the sequence in flight
    bool inter = false;
    if ((w & W_STATE) == 0) return last;
    for (int64_t j = pos; j <= len; j++) {
        if (A.steps_left != nullptr && --(*A.steps_left) < 0) return OUT_OF_BUDGET;
        const uint32_t b = j < len ? fetch(j) : 0u;     // virtual trailing NUL at j == len
        if (inter && (b & 0xC0) != 0x80) {              // sequence broken: pending bytes replay as U+FFFF
            const uint32_t f = __ldg(A.flags + (w & W_STATE));
            const int pending = (int)(j - seq);
            for (int k = 1; k <= pending; k++)
                if (f & (SF_FAILACC1 << (k - 1))) last = seq + k;
            inter = false;                              // byte j starts afresh (it may itself be a lead byte)
        }
        const uint32_t nw = T.next(w & W_STATE, b);
        if ((nw & W_INTER) && !inter) seq = j;
        inter = (nw & W_INTER) != 0;
        w = nw;
        if (w & W_ACC) last = j + 1;
        if ((w & W_STATE) == 0) break;
    }
    return last;
}

// attempt from position `start` of S = NUL || text || NUL (1-based, as in the reference)
template <class TBL, class FETCH>
__device__ __forceinline__ int64_t attempt_at(const Anchored& A, const TBL& T, FETCH fetch, int64_t len, int64_t start) {
    if (start == 1) {
        if (A.start_nul == 0) return -1;
        int64_t last = (__ldg(A.flags + A.start_nul) & SF_ACC) ? 0 : -1;
        return run_attempt(A, T, fetch, len, (uint32_t)A.start_nul, 0, last);
    }
    return run_attempt(A, T, fetch, len, (uint32_t)A.q0, start - 2, -1);
}

// length of the character at `pos` under the reference's strict decoder (utf8_m.f90:168-246)
template <class FETCH>
__device__ __forceinline__ int char_len(FETCH fetch, int64_t len, int64_t pos) {
    const uint32_t b = fetch(pos);
    int n;
    if (b < 0x80) return 1;
    else if ((b >> 5) == 6) n = 2;
    else if ((b >> 4) == 14) n = 3;
    else if ((b >> 3) == 30) n = 4;
    else return 1;
    if (pos + n > len) return 1;
    for (int k = 1; k < n; k++)
        if ((fetch(pos + k) & 0xC0) != 0x80) return 1;
    return n;
}

// S(i): byte i (1-based) of NUL || text || NUL
template <class FETCH>
__device__ __forceinline__ uint32_t framed(FETCH fetch, int64_t len, int64_t i) {
    return (i <= 1 || i >= len + 2) ? 0u : fetch(i - 2);
}
// index(S(from:), lit) + from - 1, or 0 (Fortran index(): an empty literal is found at `from`)
template <class FETCH>
__device__ inline int64_t framed_index(FETCH fetch, int64_t len, const uint8_t* lit, int n, int64_t from) {
    const int64_t m = len + 2;
    for (int64_t pos = from; pos + n - 1 <= m; pos++) {
        bool eq = true;
        for (int k = 0; k < n && eq; k++) eq = framed(fetch, len, pos + k) == __ldg(lit + k);
        if (eq) return pos;
    }
    return 0;
}
// index(x, lit, back=.true.) over S (framed != 0) or over the bare text; 0 if absent
template <class FETCH>
__device__ inline int64_t index_back(FETCH fetch, int64_t len, const uint8_t* lit, int n, bool over_frame) {
    const int64_t m = over_frame ? len + 2 : len;
    if (n > m) return 0;
    for (int64_t pos = m - n + 1; pos >= 1; pos--) {
        bool eq = true;
        for (int k = 0; k < n && eq; k++)
            eq = (over_frame ? framed(fetch, len, pos + k) : fetch(pos - 1 + k)) == __ldg(lit + k);
        if (eq) return pos;
    }
    return 0;
}

// Brute-force search (api_internal_m.F90:108-155): starts = the leading NUL, then every character boundary of the
// text, in order; the first start whose anchored run accepts after >= 1 symbol wins, with its last accept as the end.
// Written as ONE flat loop -- each iteration is a single byte step of the attempt in flight -- so that the lanes of a
// warp, which are all at different starts of different strings, still execute the same instructions.
template <class TBL, class FETCH>
__device__ __forceinline__ void brute_force_flat(const Anchored& A, const TBL& T, FETCH fetch, int64_t len,
                                                 int64_t& from, int64_t& to) {
    from = 0; to = 0;
    int64_t cur = -1;          // text index of the attempt's start; -1 = the leading NUL sentinel (S position 1)
    int64_t j = 0, seq = 0, last = -1;
    uint32_t w = (uint32_t)A.start_nul;
    bool inter = false;
    if (A.start_nul != 0) {
        last = (__ldg(A.flags + A.start_nul) & SF_ACC) ? 0 : -1;
    } else {
        if (len == 0) return;
        cur = 0;
        w = (uint32_t)A.q0;
    }
    while (true) {
        if (A.steps_left != nullptr && --(*A.steps_left) < 0) { from = -2; to = -2; return; }
        const uint32_t b = j < len ? fetch(j) : 0u;     // virtual trailing NUL at j == len
        if (inter && (b & 0xC0) != 0x80) {              // sequence broken: pending bytes replay as U+FFFF
            const uint32_t f = __ldg(A.flags + (w & W_STATE));
            const int pending = (int)(j - seq);
            for (int k = 1; k <= pending; k++)
                if (f & (SF_FAILACC1 << (k - 1))) last = seq + k;
            inter = false;
        }
        const uint32_t nw = T.next(w & W_STATE, b);
        if ((nw & W_INTER) && !inter) seq = j;
        inter = (nw & W_INTER) != 0;
        w = nw;
        j++;
        if (w & W_ACC) last = j;
        if ((w & W_STATE) == 0 || j > len) {            // this attempt is over
            if (last >= 0) {
                const int64_t e = last < len ? last : len;
                if (cur < 0) { if (e > 0) { from = 1; to = e; } }   // the NUL start wins even with an empty span
                else { from = cur + 1; to = e; }
                return;
            }
            cur = cur < 0 ? 0 : cur + char_len(fetch, len, cur);
            if (cur >= len) return;
            w = (uint32_t)A.q0;
            j = cur;
            last = -1;
            inter = false;
        }
    }
}

// brute_force_flat specialised for a string that sits in shared memory (32-bit indices, no functor): the hot form
// of K3.  Same semantics, leaner loop.  (Measured on C3: the work per string varies ~3x between the lanes of a warp
// -- it depends on where, or whether, the string matches -- so a warp averages ~10 busy lanes; claiming strings
// dynamically per lane and a warp-vote loop were both tried and gave no gain.  See DESIGN.md section 5.)
template <class TBL>
__device__ __forceinline__ void brute_force_smem(const Anchored& A, const TBL& T, uint32_t a, int len,
                                                 int64_t& from, int64_t& to) {
    from = 0; to = 0;
    int cur = -1;              // start of the attempt in flight (-1: the leading NUL sentinel)
    int j = 0, seq = 0, last = -1;
    uint32_t w = (uint32_t)A.start_nul;
    bool inter = false;
    if (A.start_nul != 0) {
        last = (__ldg(A.flags + A.start_nul) & SF_ACC) ? 0 : -1;
    } else {
        cur = 0;
        w = (uint32_t)A.q0;
    }
    const uint32_t q0 = (uint32_t)A.q0;
    while (true) {
        const uint32_t b = j < len ? lds_u8(a + j) : 0u;     // virtual trailing NUL at j == len
        if (inter && (b & 0xC0) != 0x80) {                   // sequence broken: pending bytes replay as U+FFFF
            const uint32_t f = __ldg(A.flags + (w & W_STATE));
            for (int k = 1; k <= j - seq; k++)
                if (f & (SF_FAILACC1 << (k - 1))) last = seq + k;
            inter = false;
        }
        const uint32_t nw = T.next(w & W_STATE, b);
        if ((nw & W_INTER) && !inter) seq = j;
        inter = (nw & W_INTER) != 0;
        w = nw;
        j++;
        if (w & W_ACC) last = j;
        if ((w & W_STATE) == 0 || j > len) {                 // this attempt is over
            if (last >= 0) {
                const int e = last < len ? last : len;
                if (cur < 0) { if (e > 0) { from = 1; to = e; } }
                else { from = cur + 1; to = e; }
                return;
            }
            if (cur < 0) cur = 0;
            else {
                const uint32_t c0 = lds_u8(a + cur);
                int n = 1;
                if (c0 >= 0xC0 && c0 < 0xF8) {               // lead byte: the character is n bytes only if well formed
                    n = c0 < 0xE0 ? 2 : c0 < 0xF0 ? 3 : 4;
                    bool ok = cur + n <= len;
                    if (ok) ok = (lds_u8(a + cur + 1) & 0xC0) == 0x80;
                    if (ok && n > 2) ok = (lds_u8(a + cur + 2) & 0xC0) == 0x80;
                    if (ok && n > 3) ok = (lds_u8(a + cur + 3) & 0xC0) == 0x80;
                    if (!ok) n = 1;
                }
                cur += n;
            }
            if (cur >= len) return;
            w = q0;
            j = cur;
            last = -1;
            inter = false;
        }
    }
}

// ---- NFA engine: patterns whose eager automaton passes the state cap -------------------------------------
// The reference's own per-character step (automaton%construct, src/automaton_m.F90:333-381: reachable set, epsilon
// closure) on bit sets: cur' = OR over s in cur of trans[s][class(symbol)], closures precomputed by the host.  One
// thread per text; sets live in local memory.  Same drivers as the table engine: attempt_at / brute_force_flat are
// overloaded on the engine type, so including_exact / eval_regex below serve both.
static constexpr int NFA_MAX_WORDS = 128;        // 8191 NFA states
struct NfaEngine {
    const uint64_t* trans;      // (nstates + 1) x nclasses x words
    const uint64_t* q0;         // closure(entry)
    const int32_t* cuts;        // nclasses + 1 ascending code points
    int words, nclasses, exit_state, nul_class, ffff_class, q0_accepting;
};
__device__ inline int nfa_class(const NfaEngine& N, uint32_t cp) {
    int lo = 0, hi = N.nclasses;               // largest c with cuts[c] <= cp  (cuts[nclasses] is past every code point)
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if ((uint32_t)__ldg(N.cuts + mid) <= cp) lo = mid; else hi = mid;
    }
    return lo;
}
// cur <- step(cur, class c); returns false when the result is empty
__device__ inline bool nfa_step(const NfaEngine& N, uint64_t* cur, uint64_t* nxt, int c) {
    for (int w = 0; w < N.words; w++) nxt[w] = 0;
    for (int w = 0; w < N.words; w++) {
        uint64_t bits = cur[w];
        while (bits) {
            const int s = (w << 6) + __ffsll((long long)bits) - 1;
            bits &= bits - 1;
            const uint64_t* row = N.trans + ((size_t)s * (size_t)N.nclasses + (size_t)c) * (size_t)N.words;
            for (int k = 0; k < N.words; k++) nxt[k] |= __ldg(row + k);
        }
    }
    bool any = false;
    for (int w = 0; w < N.words; w++) { cur[w] = nxt[w]; any = any || nxt[w] != 0; }
    return any;
}
__device__ __forceinline__ bool nfa_accepting(const NfaEngine& N, const uint64_t* cur) {
    return (cur[N.exit_state >> 6] >> (N.exit_state & 63)) & 1ull;
}
// the symbol at text index j under the reference's strict decoder: class and length in bytes
template <class FETCH>
__device__ inline int nfa_symbol(const NfaEngine& N, FETCH fetch, int64_t len, int64_t j, int& nbytes) {
    const uint32_t b = fetch(j);
    nbytes = char_len(fetch, len, j);
    if (b < 0x80) return nfa_class(N, b);
    if (nbytes == 1) return N.ffff_class;      // stray or malformed byte: U+FFFF (api_internal_m.F90:129-133)
    uint32_t cp = nbytes == 2 ? (b & 0x1Fu) : nbytes == 3 ? (b & 0x0Fu) : (b & 0x07u);
    for (int k = 1; k < nbytes; k++) cp = (cp << 6) | (fetch(j + k) & 0x3Fu);
    return nfa_class(N, cp);
}
// attempt from position `start` of S = NUL || text || NUL: same contract as the table engine's attempt_at
template <class FETCH>
__device__ inline int64_t attempt_at(const Anchored&, const NfaEngine& N, FETCH fetch, int64_t len, int64_t start) {
    uint64_t cur[NFA_MAX_WORDS], nxt[NFA_MAX_WORDS];
    for (int w = 0; w < N.words; w++) cur[w] = __ldg(N.q0 + w);
    int64_t last = -1, j = start - 2;
    if (start == 1) {
        if (!nfa_step(N, cur, nxt, N.nul_class)) return -1;
        if (nfa_accepting(N, cur)) last = 0;
        j = 0;
    }
    while (j <= len) {
        int nb = 1;
        const int c = j < len ? nfa_symbol(N, fetch, len, j, nb) : N.nul_class;      // virtual trailing NUL at j == len
        if (!nfa_step(N, cur, nxt, c)) break;
        j += nb;
        if (nfa_accepting(N, cur)) last = j;
    }
    return last;
}
// the brute-force search (api_internal_m.F90:108-155): the leading NUL, then every character boundary, in order
template <class FETCH>
__device__ inline void brute_force_flat(const Anchored& A, const NfaEngine& N, FETCH fetch, int64_t len, int64_t& from, int64_t& to) {
    from = 0; to = 0;
    int64_t last = attempt_at(A, N, fetch, len, 1);
    if (last >= 0) { const int64_t e = last < len ? last : len; if (e > 0) { from = 1; to = e; } return; }
    for (int64_t cur = 0; cur < len; cur += char_len(fetch, len, cur)) {
        last = attempt_at(A, N, fetch, len, cur + 2);
        if (last >= 0) { from = cur + 1; to = last < len ? last : len; return; }
    }
}
// do_matching_exactly's walk (api_internal_m.F90:247-298; SURVEY Q5) on the NFA
template <class FETCH>
__device__ inline bool nfa_match(const NfaEngine& N, FETCH fetch, int64_t len) {
    if (len == 0) return N.q0_accepting != 0;
    uint64_t cur[NFA_MAX_WORDS], nxt[NFA_MAX_WORDS], keep[NFA_MAX_WORDS];
    for (int w = 0; w < N.words; w++) { cur[w] = __ldg(N.q0 + w); keep[w] = cur[w]; }
    if (!nfa_step(N, cur, nxt, N.nul_class))                  // the leading NUL has no transition: skipped (:280-289)
        for (int w = 0; w < N.words; w++) cur[w] = keep[w];
    for (int64_t j = 0; j < len; ) {
        int nb = 1;
        const int c = nfa_symbol(N, fetch, len, j, nb);
        if (!nfa_step(N, cur, nxt, c)) return false;
        j += nb;
    }
    if (nfa_accepting(N, cur)) return true;
    return nfa_step(N, cur, nxt, N.nul_class) && nfa_accepting(N, cur);
}

// do_matching_including for a non-blank text (api_internal_m.F90:76-164): candidate starts are either
// every character boundary (no usable prefix) or the non-overlapping occurrences of the extracted
// prefix in S (utility_m.f90:58-117), cut short by the last occurrence of the extracted suffix.
// Writes the reference's (from, to) before the wrapper's `from>0 .and. to>0` test.
template <class TBL, class FETCH>
__device__ inline void including_exact(const Anchored& A, const TBL& T, FETCH fetch, int64_t len,
                                       const uint8_t* pre, int pre_len, bool pre_active,
                                       const uint8_t* suf, int suf_len, bool suf_active,
                                       int64_t& from, int64_t& to) {
    const int64_t NONE = -9999;
    const int64_t m = len + 2;
    from = 0; to = 0;
    bool brute = !pre_active;
    int64_t first = NONE, frame_suf = NONE, offset = 0;
    bool more = false;
    if (!brute) {
        const int64_t idx = framed_index(fetch, len, pre, pre_len, 1);
        frame_suf = index_back(fetch, len, suf, suf_len, true);
        if (frame_suf == 0) frame_suf = NONE;
        if (idx > 0) {
            if (frame_suf != NONE) { if (idx <= frame_suf) first = idx; }
            else first = idx;
            offset = idx + pre_len - 1;
            more = true;
        }
        if (first == NONE) brute = true;
    }
    if (brute) { brute_force_flat(A, T, fetch, len, from, to); return; }
    bool at_zero = first == 2;                 // "i = 0": try the leading NUL before the first occurrence
    int64_t start = at_zero ? 1 : first;
    int64_t text_suf = NONE;
    if (suf_active) {
        text_suf = index_back(fetch, len, suf, suf_len, false);
        if (text_suf == 0) return;
    }
    while (start < m) {
        if (text_suf != NONE && text_suf < start) return;
        const int64_t last = attempt_at(A, T, fetch, len, start);
        if (last == OUT_OF_BUDGET) { from = -2; to = -2; return; }
        if (last >= 0) {
            from = start - 1 < 1 ? 1 : start - 1;
            to = last < len ? last : len;      // max_match >= len(str) -> len(string), else max_match - 2
            return;
        }
        if (at_zero) { at_zero = false; start = first; continue; }
        if (!more || !(offset < m)) return;
        const int64_t hit = framed_index(fetch, len, pre, pre_len, offset + 1);
        if (hit <= 0) return;
        start = hit;
        offset = hit + pre_len - 1;            // offset + idx + len_pre - 1 with idx = hit - offset
        if (frame_suf != NONE && offset > frame_suf) more = false;
    }
}

// `.in.` through the exact prefix-candidate search (pattern has a non-blank prefix, `all` is blank)
template <class FETCH>
__device__ inline bool in_with_prefix(const KParams& p, FETCH fetch, int64_t len) {
    if (len == 0 || (len == 1 && fetch(0) == 0x20)) return p.q0_accepting != 0;
    Table<3> T;
    T.g_table = p.a_table; T.g_cmap = p.a_classmap; T.shift = p.a_row_shift; T.s_table = 0; T.s_cmap = 0;
    Anchored A{p.a_flags, p.a_start_nul, p.a_q0};
    int64_t f, t;
    including_exact(A, T, fetch, len, p.lits + p.all_len, p.pre_len, p.pre_active != 0,
                    p.lits + p.all_len + p.pre_len, p.suf_len, p.suf_active != 0, f, t);
    return f > 0 && t > 0;
}

// full regex() semantics for one text; writes Forgex's (from, to) (0,0 = no match)
template <class TBL, class FETCH>
__device__ inline void eval_regex(const KParams& p, const TBL& T, FETCH fetch, int64_t len, int64_t& from, int64_t& to) {
    from = 0; to = 0;
    if (p.all_active) {  // literal fast path (forgex.F90:281-307)
        const int n = p.all_len;
        for (int64_t i = 0; i + n <= len; i++) {
            bool eq = true;
            for (int k = 0; k < n && eq; k++) eq = fetch(i + k) == __ldg(p.lits + k);
            if (eq) { from = i + 1; to = i + n; return; }
        }
        return;
    }
    if (len == 0 || (len == 1 && fetch(0) == 0x20)) return;      // api_internal_m.F90:68-74 -> '' / 0 / 0
    Anchored A{p.flags, p.start_nul, p.q0};
    A.steps_left = p.steps_left;
    int64_t f, t;
    including_exact(A, T, fetch, len, p.lits + p.all_len, p.pre_len, p.pre_active != 0,
                    p.lits + p.all_len + p.pre_len, p.suf_len, p.suf_active != 0, f, t);
    if (f == -2) { from = -2; to = -2; return; }                 // out of work budget (k_buffer_sequential only)
    if (f > 0 && t > 0) { from = f; to = t; }                    // forgex.F90:332-343
}

// ---- slow path: full wrapper semantics incl. literal gates, text read from global memory ------------
// Kept out of line so that the hot loops stay small.  Uses the class-compressed table in global memory.
__device__ __forceinline__ bool lit_equal(const uint8_t* a, const uint8_t* lit, int n) {
    for (int i = 0; i < n; i++) if (__ldg(a + i) != __ldg(lit + i)) return false;
    return true;
}
// index(text, lit): 1-based position of the first occurrence, 0 if none (forgex.F90:114, :284)
__device__ inline int64_t lit_index(const uint8_t* s, int64_t len, const uint8_t* lit, int n) {
    if (n > len) return 0;
    if (n == 0) return 1;
    for (int64_t i = 0; i + n <= len; i++)
        if (lit_equal(s + i, lit, n)) return i + 1;
    return 0;
}

template <int OP>
__device__ __noinline__ bool eval_bool_slow(const KParams& p, const uint8_t* s, int64_t len) {
    const uint8_t* all = p.lits;
    const uint8_t* pre = p.lits + p.all_len;
    const uint8_t* suf = pre + p.pre_len;
    if (OP == 1) {
        if (p.all_active) return lit_index(s, len, all, p.all_len) > 0;
        if (p.prefix_mode == 2) return in_with_prefix(p, FetchGlobal{s}, len);
    } else {
        if (p.all_active && len == p.all_len) return lit_equal(s, all, p.all_len);
        // prefix / suffix gate of do_matching_exactly (api_internal_m.F90:199-233)
        int64_t lp = p.pre_len, ls = p.suf_len;
        if (len > 0 && lp > 0 && lp == len && lit_equal(s, pre, (int)lp)) return true;
        if (lp > len || ls > len) return false;
        if (len > 0) {
            if (p.pre_active && !lit_equal(s, pre, (int)lp)) return false;
            if (p.suf_active && !lit_equal(s + (len - ls), suf, (int)ls)) return false;
        } else {
            if (p.pre_active && lp != 0) return false;
            if (p.suf_active && ls != 0) return false;
        }
    }
    if (degenerate_text<OP>(len, len ? __ldg(s) : 0)) return p.q0_accepting != 0;
    Table<3> T;
    T.g_table = p.ctable; T.g_cmap = p.classmap; T.shift = p.c_row_shift; T.s_table = 0; T.s_cmap = 0;
    uint32_t st = (uint32_t)p.start;
    uint32_t high = 0;
    for (int64_t i = 0; i < len; i++) { uint32_t b = __ldg(s + i); high |= b; st = T.next(st, b); }
    bool r = result_flag(p, st);
    if (OP == 1 && r && p.prefix_mode == 1 && (high & 0x80)) r = in_with_prefix(p, FetchGlobal{s}, len);
    return r;
}
__device__ __noinline__ bool recheck_in_with_prefix(const KParams& p, const uint8_t* s, int64_t len) {
    return in_with_prefix(p, FetchGlobal{s}, len);
}

template <int KIND>
__device__ __forceinline__ uint32_t step4(const Table<KIND>& T, uint32_t st, uint32_t w) {
    st = T.next(st, w & 0xFF);
    st = T.next(st, (w >> 8) & 0xFF);
    st = T.next(st, (w >> 16) & 0xFF);
    st = T.next(st, w >> 24);
    return st;
}

// offsets of a ragged batch as the host handed them over: ascending, first 0, none past `total`?  (*bad != 0 if not.)
// The host-pointer entry points run this before any kernel reads text through those offsets.
__global__ void k_check_offsets(const int64_t* __restrict__ off, int64_t n, int64_t total, int* __restrict__ bad) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    bool wrong = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t a = __ldg(off + i), b = __ldg(off + i + 1);
        wrong |= a > b || a < 0 || b > total;
    }
    if (wrong) *bad = 1;
}

// ---------------------------------------------------------------------------------------------
// K1: fixed-stride batch, boolean result (configs C1 `.match.` 8-byte strings, C5 `.in.` 64-byte)
// One thread per string; consecutive threads read consecutive strings, so a warp's loads cover a
// contiguous 32*stride-byte span.
// ---------------------------------------------------------------------------------------------
template <int OP, int KIND, int VEC>
__global__ void __launch_bounds__(256) k_bool_fixed(KParams p, const uint8_t* __restrict__ buf, int64_t n, int64_t stride,
                                                    uint8_t* __restrict__ out, int generic) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_cmap = smem;
    uint8_t* s_table = smem + 256;
    Table<KIND> T = stage_table<KIND>(p, s_table, s_cmap);
    if (KIND != 3) __syncthreads();
    const int64_t gstride = (int64_t)gridDim.x * blockDim.x;
    if ((VEC == 8 || VEC == 16) && !generic && stride == VEC) {
        // One load covers a whole string (C1: 8 bytes): the walk is 8-16 lookups, short against the latency of the load
        // in front of it, so a thread takes FOUR strings per step -- all loads first, then the four walks.  The four are
        // a grid stride apart: every load instruction of a warp reads one contiguous run and every store instruction
        // writes one whole sector.  (Tried: four CONSECUTIVE strings per thread and one 4-byte store -- the loads then
        // touch each sector four times, DRAM read traffic 1.19x, 338 vs 298 us per GiB.)
        for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += 4 * gstride) {
            constexpr int NW = VEC == 16 ? 4 : 2;          // 32-bit words per string
            uint32_t w[4][NW];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int64_t i = i0 + u * gstride;
#pragma unroll
                for (int q = 0; q < NW; q++) w[u][q] = 0;
                if (i < n) {
                    if (VEC == 16) { const uint4 v = ldg_nc_v4(buf + i * stride); w[u][0] = v.x; w[u][1] = v.y; w[u][NW - 2] = v.z; w[u][NW - 1] = v.w; }
                    else { const uint2 v = ldg_nc_v2(buf + i * stride); w[u][0] = v.x; w[u][1] = v.y; }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int64_t i = i0 + u * gstride;
                if (i < n) {
                    uint32_t st = (uint32_t)p.start, high = 0;
#pragma unroll
                    for (int q = 0; q < NW; q++) { high |= w[u][q]; st = step4(T, st, w[u][q]); }
                    bool r = result_flag(p, st);
                    if (OP == 1 && r && p.prefix_mode == 1 && (high & 0x80808080u)) r = recheck_in_with_prefix(p, buf + i * stride, stride);
                    out[i] = r ? 1 : 0;
                }
            }
        }
        return;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gstride) {
        const uint8_t* s = buf + i * stride;
        bool r;
        if (generic) {
            r = eval_bool_slow<OP>(p, s, stride);
        } else if (degenerate_text<OP>(stride, stride ? __ldg(s) : 0)) {
            r = p.q0_accepting != 0;
        } else {
            uint32_t st = (uint32_t)p.start;
            uint32_t high = 0;
            if (VEC == 16) {
                for (int64_t k = 0; k < stride; k += 16) {
                    uint4 v = ldg_nc_v4(s + k);
                    high |= v.x | v.y | v.z | v.w;
                    st = step4(T, st, v.x); st = step4(T, st, v.y); st = step4(T, st, v.z); st = step4(T, st, v.w);
                }
            } else if (VEC == 8) {
                for (int64_t k = 0; k < stride; k += 8) {
                    uint2 v = ldg_nc_v2(s + k);
                    high |= v.x | v.y;
                    st = step4(T, st, v.x); st = step4(T, st, v.y);
                }
            } else {
                for (int64_t k = 0; k < stride; k++) { uint32_t b = __ldg(s + k); high |= b; st = T.next(st, b); }
            }
            r = result_flag(p, st);
            if (OP == 1 && r && p.prefix_mode == 1 && (high & 0x80808080u)) r = recheck_in_with_prefix(p, s, stride);
        }
        out[i] = r ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------------------------
// K1c: fixed-stride batch, boolean result, BIG automaton with a small ASCII alphabet (config C5: 10252 states, but the
// ASCII bytes fall into three classes -- a, b, everything else).  The class-compressed table of such a pattern (16
// classes, 328 KB) fits neither shared memory nor L1; its ASCII columns alone do: 4 columns x 2 bytes = 8 bytes per
// state, 82 KB.  Strings that hold a byte >= 0x80 (multi-byte sequences need the other 12 columns) are decided by the
// full table (eval_bool_slow); everything else walks the compact one -- from shared memory (SMEM), or, when the caller
// forces the global path (BASELINE config 5 is stated as the L2/HBM table path), from global memory, where 82 KB stay
// in L1 and four rows share a 32-byte sector.  The byte -> column map is a 256-byte table in shared memory either way.
// ---------------------------------------------------------------------------------------------
template <int OP, bool SMEM>
__global__ void __launch_bounds__(1024, 2) k_bool_fixed_compact(KParams p, const uint16_t* __restrict__ ctab, const uint8_t* __restrict__ cmap4,
                                                               const uint8_t* __restrict__ buf, int64_t n, int64_t stride,
                                                               uint8_t* __restrict__ out) {
    extern __shared__ __align__(128) uint8_t smem[];
    for (int i = threadIdx.x; i < 64; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = __ldg(reinterpret_cast<const uint32_t*>(cmap4) + i);
    if (SMEM)
        for (int i = threadIdx.x; i < p.nstates * 2; i += blockDim.x)
            reinterpret_cast<uint32_t*>(smem + 256)[i] = __ldg(reinterpret_cast<const uint32_t*>(ctab) + i);
    __syncthreads();
    const uint32_t s_cmap = smem_u32(smem), s_tab = smem_u32(smem + 256);
    auto next = [&](uint32_t st, uint32_t byte) -> uint32_t {
        const uint32_t c = lds_u8(s_cmap + byte);
        return SMEM ? lds_u16(s_tab + st * 8 + c * 2) : (uint32_t)__ldg(ctab + st * 4 + c);
    };
    const int64_t gstride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gstride) {
        const uint8_t* s = buf + i * stride;
        uint32_t st = (uint32_t)p.start, high = 0;
        int64_t k = 0;
        for (; k + 32 <= stride; k += 32) {            // a whole 32-byte sector per step: both halves asked for back to back
            const uint4 v0 = ldg_nc_v4(s + k), v1 = ldg_nc_v4(s + k + 16);
            high |= v0.x | v0.y | v0.z | v0.w | v1.x | v1.y | v1.z | v1.w;
            const uint32_t w[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
            for (int q = 0; q < 8; q++) {
                st = next(st, w[q] & 0xFFu);
                st = next(st, (w[q] >> 8) & 0xFFu);
                st = next(st, (w[q] >> 16) & 0xFFu);
                st = next(st, w[q] >> 24);
            }
        }
        for (; k < stride; k += 16) {
            const uint4 v = ldg_nc_v4(s + k);
            high |= v.x | v.y | v.z | v.w;
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                st = next(st, w[q] & 0xFFu);
                st = next(st, (w[q] >> 8) & 0xFFu);
                st = next(st, (w[q] >> 16) & 0xFFu);
                st = next(st, w[q] >> 24);
            }
        }
        bool r = result_flag(p, st);
        if (high & 0x80808080u) r = eval_bool_slow<OP>(p, s, stride);      // a non-ASCII byte: the full table decides
        out[i] = r ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------------------------
// K2: ragged batch (flat buffer + int64 offsets), boolean result (config C2 `.in.`)
// A CTA owns tile t = strings [t*spt, (t+1)*spt).  Their bytes are contiguous in the flat buffer, so the
// tile is brought into shared memory by ONE TMA bulk copy (up to `cap` bytes; strings that reach past the
// staged region are walked from global memory by the slow path).  The tile's offsets are staged next to it
// as 32-bit tile-relative values, each thread walks one string at a time out of shared memory, and the
// results are written back as one coalesced run.
// ---------------------------------------------------------------------------------------------
// Stage bytes [t0, t1) of buf into shared memory at `tile` such that byte x lives at tile[x - base],
// base = t0 rounded down so that the global source is 16-byte aligned.  Returns base.
__device__ __forceinline__ int64_t stage_tile(const uint8_t* __restrict__ buf, int64_t t0, int64_t t1,
                                              int64_t total, uint8_t* tile, uint32_t mbar, bool& armed) {
    const uintptr_t g0 = reinterpret_cast<uintptr_t>(buf) + (uintptr_t)t0;
    const int64_t base = t0 - (int64_t)(g0 & 15);                       // may be < 0 by up to 15 (stays inside the allocation)
    const uintptr_t gend = reinterpret_cast<uintptr_t>(buf) + (uintptr_t)total;
    uintptr_t gcopy_end = (reinterpret_cast<uintptr_t>(buf) + (uintptr_t)t1 + 15) & ~(uintptr_t)15;
    const uintptr_t gsafe_end = gend & ~(uintptr_t)15;                   // never bulk-read past the last whole 16-byte block
    if (gcopy_end > gsafe_end) gcopy_end = gsafe_end;
    const uintptr_t gsrc = g0 & ~(uintptr_t)15;
    const uint32_t bulk = gcopy_end > gsrc ? (uint32_t)(gcopy_end - gsrc) : 0u;
    armed = bulk != 0;
    if (bulk && threadIdx.x == 0) {
        mbar_expect_tx(mbar, bulk);
        bulk_g2s(smem_u32(tile), reinterpret_cast<const void*>(gsrc), bulk, mbar);
    }
    // tail (< 16 bytes at the very end of the buffer): plain loads
    const int64_t copied_to = (int64_t)(gsrc + bulk - reinterpret_cast<uintptr_t>(buf));
    for (int64_t x = copied_to + threadIdx.x; x < t1; x += blockDim.x)
        if (x >= 0) tile[x - base] = __ldg(buf + x);
    return base;
}

template <int KIND>
__device__ __forceinline__ uint32_t walk_smem(const Table<KIND>& T, uint32_t st, uint32_t addr, int len, uint32_t& high) {
    int i = 0;
    while (i < len && ((addr + i) & 3)) { uint32_t b = lds_u8(addr + i); high |= b; st = T.next(st, b); i++; }
    for (; i + 4 <= len; i += 4) { uint32_t w = lds_u32(addr + i); high |= w; st = step4(T, st, w); }
    for (; i < len; i++) { uint32_t b = lds_u8(addr + i); high |= b; st = T.next(st, b); }
    return st;
}

static constexpr int32_t OFF_BEYOND = 0x7FFFFFFF;   // staged offset of a position past the staged bytes

// common tile prologue of K2 / K3: stages text + offsets of tile t
struct TileCtx {
    int64_t first;     // first string of the tile
    int count;         // strings in the tile
    int64_t base;      // buffer position of tile[0]
    int64_t t1;        // end of the staged bytes (buffer position)
};
__device__ __forceinline__ TileCtx load_tile(const uint8_t* __restrict__ buf,
                                             const int64_t* __restrict__ offsets, int64_t n, int64_t total, int64_t t,
                                             int spt, int cap, uint8_t* tile, int32_t* s_off, uint32_t mbar,
                                             uint32_t& phase) {
    TileCtx c;
    c.first = t * spt;
    c.count = (int)((n - c.first) < spt ? (n - c.first) : spt);
    const int64_t t0 = __ldg(offsets + c.first);
    const int64_t tend = __ldg(offsets + c.first + c.count);
    c.t1 = tend - t0 > cap ? t0 + cap : tend;
    bool armed = false;
    c.base = t0;
    if (t0 < c.t1) c.base = stage_tile(buf, t0, c.t1, total, tile, mbar, armed);
    for (int i = threadIdx.x; i <= c.count; i += blockDim.x) {          // overlaps with the bulk copy in flight
        const int64_t o = __ldg(offsets + c.first + i);
        s_off[i] = o > c.t1 ? OFF_BEYOND : (int32_t)(o - c.base);
    }
    if (armed) { mbar_wait(mbar, phase); phase ^= 1; }
    __syncthreads();
    return c;
}

// shared-memory layout of the ragged kernels (must match make_tiling() in fx_cabi.cu):
//   [0,16) mbarrier | classmap 256 | table | offsets (spt+4) x int32 | results spt | pad to 128 | tile (cap+64)
__host__ __device__ __forceinline__ int tile_offset(int table_smem_bytes, int spt) {
    return (16 + 256 + table_smem_bytes + (spt + 4) * 4 + spt + 127) & ~127;
}

template <int OP, int KIND>
__global__ void __launch_bounds__(256, 4) k_bool_ragged(KParams p, const uint8_t* __restrict__ buf,
                                                        const int64_t* __restrict__ offsets, int64_t n, int64_t total,
                                                        uint8_t* __restrict__ out, int spt, int cap, int64_t ntiles,
                                                        int table_smem_bytes, int generic) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_cmap = smem + 16;
    uint8_t* s_table = smem + 16 + 256;
    int32_t* s_off = reinterpret_cast<int32_t*>(smem + 16 + 256 + table_smem_bytes);
    uint8_t* s_res = reinterpret_cast<uint8_t*>(s_off + spt + 4);
    uint8_t* tile = smem + tile_offset(table_smem_bytes, spt);
    const uint32_t mbar = smem_u32(smem);
    Table<KIND> T = stage_table<KIND>(p, s_table, s_cmap);
    if (threadIdx.x == 0) mbar_init(mbar, 1);
    __syncthreads();
    uint32_t phase = 0;
    const uint32_t tile_addr = smem_u32(tile);
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const TileCtx c = load_tile(buf, offsets, n, total, t, spt, cap, tile, s_off, mbar, phase);
        for (int i = threadIdx.x; i < c.count; i += blockDim.x) {
            const int32_t r0 = s_off[i], r1 = s_off[i + 1];
            bool r;
            if (generic || r1 == OFF_BEYOND) {
                const int64_t o0 = __ldg(offsets + c.first + i), o1 = __ldg(offsets + c.first + i + 1);
                r = eval_bool_slow<OP>(p, buf + o0, o1 - o0);
            } else {
                const int len = r1 - r0;
                const uint32_t a = tile_addr + (uint32_t)r0;
                if (degenerate_text<OP>(len, len ? lds_u8(a) : 0)) r = p.q0_accepting != 0;
                else {
                    uint32_t high = 0;
                    r = result_flag(p, walk_smem(T, (uint32_t)p.start, a, len, high));
                    if (OP == 1 && r && p.prefix_mode == 1 && (high & 0x80808080u))
                        r = recheck_in_with_prefix(p, buf + (c.base + r0), len);
                }
            }
            s_res[i] = r ? 1 : 0;
        }
        __syncthreads();                 // results complete; everyone is done with the tile
        for (int i = threadIdx.x; i < c.count; i += blockDim.x) out[c.first + i] = s_res[i];
        __syncthreads();                 // before the next tile overwrites offsets / results / text
    }
}

// ---------------------------------------------------------------------------------------------
// K2c: ragged batch, boolean `.in.`, sparse starts.
// `.in.` is true when SOME start of the brute-force search wins (api_internal_m.F90:108-155).  A start whose first
// byte kills the anchored automaton cannot win, so when the set F of first bytes that survive the step out of q0 is
// small (a few byte ranges: 'f' for foo(bar|baz); NUL/LF/CR for ^ERROR...), almost every position of the text is
// ruled out by a compare.  The kernel therefore does not walk the strings at all, it has no block-wide step, and
// the text never passes through shared memory:
//   S  sweep: a warp owns tiles of consecutive strings (about 24 KB of text).  Its lanes read the tile's bytes
//      LINEARLY, 32 bytes per lane and step, as coalesced 16-byte loads straight from global memory (four rows = 4 KB
//      per warp in flight), and test them against F with SWAR arithmetic (3-4 integer instructions per 4 bytes).
//      When the automaton has ONE first byte and ONE possible second byte (a pattern that begins with a literal), the
//      test is for that byte pair.  32-byte units that pass are queued;
//   U  units: whenever 32 units are waiting, the lanes take one each (its bytes are in L2 now): every candidate
//      takes its first table step and, unless that already accepts or enters a multi-byte sequence, the second one
//      (with the next text byte, and with the NUL that would end the string there).  Two bytes kill almost every
//      candidate; survivors are queued as starts;
//   A  starts: whenever 32 starts are waiting, the lanes run them side by side: binary search over the tile's
//      offsets for the string, then the anchored attempt -- the reference's own inner loop, on the anchored
//      flag-bit table -- until the first counted accept, which sets the string's result.
// The per-string part (degenerate texts, the start on the leading NUL) is one string per lane and writes the
// tile's results before any start of that tile can run.  Every phase has all 32 lanes doing the same work whatever
// the string lengths are.
//
// Preconditions (checked on the host, fx_cabi.cu sparse_first_set): F holds no continuation byte 0x80..0xBF --
// ASCII, lead and invalid bytes always sit on a character boundary of the reference's decoder, so every candidate is
// a legal start; the start on the leading NUL is not accepting by itself, so no start can "win with an empty span"
// and stop the search early; the prefix prefilter is absent or neutral (prefix_mode 0/1; for mode 1 a winning string
// from a tile that holds bytes >= 0x80 is re-checked exactly, as in K2).
// ---------------------------------------------------------------------------------------------
struct SparseParams {
    const uint16_t* table;      // anchored flag-bit table, class-compressed
    const uint8_t* classmap;
    const uint8_t* flags;
    int table_words, row_shift, q0, start_nul;
    // ASCII range r of the sweep filter, 7-bit bounds folded into SWAR addends
    uint32_t add_lo[4];         // (0x80 - lo) * 0x01010101: bit 7 of (y + add_lo) <=> y >= lo   (NR = -1: value * 0x01010101)
    uint32_t add_hi[4];         // (0x7F - hi) * 0x01010101: bit 7 of (y + add_hi) <=> y >  hi
    uint32_t second;            // TWO: the one ASCII byte that keeps the automaton alive after the first, in all four bytes
    uint32_t second_high;       // TWO: 0xFFFFFFFF when bytes >= 0xC0 keep it alive as well (lead bytes), else 0
};

// shared memory of K2c: classmap 256 | table | pad to 16 | 8 warps x (unit queue 64 x uint4 | start queue 64 x uint4)
//   queue entry = {tile, kind | high << 31, low word, high word}
//   in front of the queues: copies of the kernel parameters (KParams, SparseParams) and one SparseCtx per warp, for the
//   out-of-line phases -- handed to them by reference from the kernel's parameter space they would be copied to every
//   thread's local memory and read back through L1/L2 (measured: +20 % DRAM traffic)
static constexpr int SPARSE_WARP_BYTES = 2 * 64 * 16;
static constexpr int SPARSE_PARAM_BYTES = 1024;
__host__ __device__ __forceinline__ int sparse_shared_head(int table_smem_bytes) { return ((256 + table_smem_bytes + 15) & ~15) + SPARSE_PARAM_BYTES; }

// Sweep filter for one 4-byte word: bit 7 set in every byte of w that may be in F (callers mask with 0x80808080).
// A superset is fine -- every candidate is confirmed by the first table step before anything else happens -- so bit 7
// of the text byte is ignored here (a byte >= 0x80 whose low bits fall into a range is a false candidate, in
// non-ASCII text only), and with HIGH every byte >= 0x80 passes (F holds lead bytes: e.g. the overlong forms 0xC1 0xE0
// 0xF0 of an ASCII first character, which the reference's structural decoder accepts).
// NR = -1: F's ASCII part is ONE byte value (add_lo[0] holds it in all four bytes): the zero-byte test on w ^ value,
//          three instructions per word (its false positives sit above a true hit, in the same word).
template <int NR, bool HIGH>
__device__ __forceinline__ uint32_t first_mask(const SparseParams& sp, uint32_t w) {
    uint32_t m = 0;
    if (NR == -1) {
        const uint32_t x = w ^ sp.add_lo[0];
        m = (x - 0x01010101u) & ~x;
    } else {
        const uint32_t y = w & 0x7F7F7F7Fu;
#pragma unroll
        for (int r = 0; r < NR; r++) m |= (y + sp.add_lo[r]) & ~(y + sp.add_hi[r]);
    }
    if (HIGH) m |= w;
    return m;
}
// TWO: the bytes of w that may follow the first byte turn into zero bytes: the second byte, and, when lead bytes can
// follow (second_high), every byte >= 0x80.  The PRMT selector of lead_sel() replicates each byte's bit 7 over the
// byte (0xBA98), or gives zero (0x4444 picks the zero operand's byte 0).
__device__ __forceinline__ uint32_t lead_sel(const SparseParams& sp) { return sp.second_high ? 0xBA98u : 0x4444u; }
template <bool LEAD>
__device__ __forceinline__ uint32_t second_zero(const SparseParams& sp, uint32_t w, uint32_t sel) {
    uint32_t z = w ^ sp.second;
    if (LEAD) {
        uint32_t s;
        asm("prmt.b32 %0, %1, 0, %2;" : "=r"(s) : "r"(w), "r"(sel));
        z &= ~s;
    }
    return z;
}
// TWO: bit 7 of byte j set when byte j of w is the first byte and the byte after it may follow: z = second_zero of
// w, z_next = second_zero of the word after w (only its byte 0 is used).  Byte j of t is zero exactly for such a
// pair; the zero-byte test also flags a 0x01 byte of t above a zero byte (a borrow neighbour), so a word with a pair
// is always flagged and a word without one never is.
__device__ __forceinline__ uint32_t pair_mask(const SparseParams& sp, uint32_t w, uint32_t z, uint32_t z_next) {
    const uint32_t t = (w ^ sp.add_lo[0]) | __funnelshift_r(z, z_next, 8);
    return (t - 0x01010101u) & ~t;
}
// Sweep filter for one 32-byte unit: non-zero when the unit may hold a candidate.  TWO (with NR = -1): a candidate
// is the first byte FOLLOWED BY the second byte (or by a lead byte, if lead bytes can follow); z_next is second_zero
// of the word after the unit (0 where that word is not known: the byte after the unit is assumed to match).  `seen`
// collects the OR of the unit's words (bytes >= 0x80 in the tile?).
template <int NR, bool HIGH, bool TWO>
__device__ __forceinline__ uint32_t unit_any(const SparseParams& sp, const uint4& a, const uint4& b, uint32_t& seen,
                                             uint32_t z_next = 0u) {
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    const uint32_t all = w[0] | w[1] | w[2] | w[3] | w[4] | w[5] | w[6] | w[7];
    seen |= all;
    uint32_t any = 0;
    if (TWO) {
        const uint32_t sel = lead_sel(sp);
#pragma unroll
        for (int k = 7; k >= 0; k--) {
            // with HIGH every byte >= 0x80 makes the unit pass anyway: lead bytes inside the unit need no test
            const uint32_t z = second_zero<!HIGH>(sp, w[k], sel);
            any |= pair_mask(sp, w[k], z, z_next);
            z_next = z;
        }
        if (HIGH) any |= all;
    } else {
#pragma unroll
        for (int k = 0; k < 8; k++) any |= first_mask<NR, false>(sp, w[k]);
        if (HIGH) any |= all;
    }
    return any & 0x80808080u;
}
// bits 7, 15, 23, 31 of m -> bits 0..3
__device__ __forceinline__ uint32_t pack_byte_flags(uint32_t m) { return ((((m >> 7) & 0x01010101u) * 0x00204081u) >> 21) & 0xFu; }

// does the anchored attempt that starts in state `st` before byte `pos` of a string of `len` bytes see a counted
// accept?  run_attempt() reduced to what a boolean needs: out at the first accept.
template <class TBL, class FETCH>
__device__ __forceinline__ bool attempt_wins(const Anchored& A, const TBL& T, FETCH fetch, int64_t len, uint32_t st, int64_t pos) {
    uint32_t w = st;
    int64_t seq = 0;
    bool inter = false;
    for (int64_t j = pos; j <= len; j++) {
        const uint32_t b = j < len ? fetch(j) : 0u;               // virtual trailing NUL at j == len
        if (inter && (b & 0xC0) != 0x80) {                        // sequence broken: pending bytes replay as U+FFFF
            const uint32_t f = __ldg(A.flags + (w & W_STATE));
            if (f & ((SF_FAILACC1 << (int)(j - seq)) - SF_FAILACC1)) return true;
            inter = false;
        }
        const uint32_t nw = T.next(w & W_STATE, b);
        if ((nw & W_INTER) && !inter) seq = j;
        inter = (nw & W_INTER) != 0;
        w = nw;
        if (w & W_ACC) return true;
        if ((w & W_STATE) == 0) return false;
    }
    return false;
}

// per-warp context of the deferred phases (everything but the queues' fill levels is read-only)
struct SparseCtx {
    const uint8_t* buf;
    const int64_t* offsets;   // nullptr: fixed-stride batch, string i = [i * stride, (i + 1) * stride)
    int64_t stride;
    uint8_t* out;
    int64_t n, total;
    int spt;
    uint4* units;     // queue of 32-byte units to look at
    uint4* starts;    // queue of starts to attempt
};
static constexpr uint32_t SPARSE_START = 0, SPARSE_RECHECK = 2;
// start of string i: from the offsets array, or i * stride for a fixed-stride batch
__device__ __forceinline__ int64_t sparse_off(const int64_t* __restrict__ offsets, int64_t stride, int64_t i) {
    return offsets ? __ldg(offsets + i) : i * stride;
}

// Phase A: `count` (<= 32) queued starts, one per lane.
//   kind SPARSE_START    {tile, kind|high, position (64 bit) relative to the tile's first byte}: find the string, attempt
//   kind SPARSE_RECHECK  {tile, kind, string number in the tile}: the string won from the leading NUL in a tile with
//                        bytes >= 0x80 and the pattern has a prefix: exact prefix replay decides
// Out of line on purpose, and called only from the outer loop of the kernel: a call inside the sweep loop makes the
// compiler keep that loop's whole state in callee-saved registers and spill it (measured: 200 bytes per thread).
template <int KIND>
__device__ __forceinline__ Table<KIND> sparse_table(const SparseParams& sp, uint32_t s_table, uint32_t s_cmap) {
    Table<KIND> T;
    T.s_table = s_table; T.s_cmap = s_cmap; T.g_table = sp.table; T.g_cmap = sp.classmap; T.shift = sp.row_shift;
    return T;
}

template <int KIND>
__device__ __noinline__ void sparse_run_starts(const KParams& p, const SparseParams& sp, uint32_t s_table, uint32_t s_cmap,
                                               const SparseCtx& c, int count) {
    const Table<KIND> T = sparse_table<KIND>(sp, s_table, s_cmap);
    const int lane = threadIdx.x & 31;
    const Anchored A{sp.flags, sp.start_nul, sp.q0};
    __syncwarp();
    if (lane < count) {
        const uint4 e = c.starts[lane];
        const int64_t first = (int64_t)e.x * c.spt;
        const int64_t* off = c.offsets + first;
        const uint32_t kind = e.y & 7u;
        const int64_t val = (int64_t)(((unsigned long long)e.w << 32) | e.z);
        if (c.offsets == nullptr) {                                // fixed stride: the string is a division away
            const int64_t s = kind == SPARSE_START ? val / c.stride : val;
            const uint8_t* str = c.buf + (first + s) * c.stride;
            bool win;
            if (kind == SPARSE_START) {
                win = !(c.stride == 1 && __ldg(str) == 0x20) &&
                      attempt_wins(A, T, FetchGlobal{str}, c.stride, (uint32_t)sp.q0, val - s * c.stride);
                if (win && p.prefix_mode == 1 && (e.y >> 31)) win = recheck_in_with_prefix(p, str, c.stride);
                if (win) c.out[first + s] = 1;
            } else {
                c.out[first + s] = recheck_in_with_prefix(p, str, c.stride) ? 1 : 0;
            }
        } else if (kind == SPARSE_START) {
            const int cnt = (int)((c.n - first) < c.spt ? (c.n - first) : c.spt);
            // largest s with off[s] <= gpos.  Interpolation search: the probes land next to the answer (one or two
            // 32-byte sectors of offsets instead of the log2(cnt) scattered ones of a bisection); bisection takes over
            // if the lengths are too uneven for that to converge
            int64_t vlo = __ldg(off), vhi = __ldg(off + cnt);
            const int64_t gpos = vlo + val;
            int s = 0, sh = cnt;
            for (int iter = 0; sh - s > 1; iter++) {
                int mid = (s + sh) >> 1;
                if (iter < 6) {
                    mid = s + (int)((float)(gpos - vlo) * (float)(sh - s) / (float)(vhi - vlo));
                    mid = mid <= s ? s + 1 : mid >= sh ? sh - 1 : mid;
                }
                const int64_t v = __ldg(off + mid);
                if (v <= gpos) { s = mid; vlo = v; } else { sh = mid; vhi = v; }
            }
            const int64_t o0 = __ldg(off + s), o1 = __ldg(off + s + 1);
            const uint8_t* str = c.buf + o0;
            if (!(o1 - o0 == 1 && __ldg(str) == 0x20)) {           // a lone blank never reaches the loop
                bool win = attempt_wins(A, T, FetchGlobal{str}, o1 - o0, (uint32_t)sp.q0, gpos - o0);
                if (win && p.prefix_mode == 1 && (e.y >> 31)) win = recheck_in_with_prefix(p, str, o1 - o0);
                if (win) c.out[first + s] = 1;
            }
        } else {
            const int64_t o0 = __ldg(off + val), o1 = __ldg(off + val + 1);
            c.out[first + val] = recheck_in_with_prefix(p, c.buf + o0, o1 - o0) ? 1 : 0;
        }
    }
    __syncwarp();
}

// Phase U: `count` (<= 32) queued units {tile, high << 31, unit number (64 bit) from the tile's 32-byte aligned base},
// one per lane.  Candidates are taken in rounds (round k = every lane's k-th candidate); a candidate survives unless
// two bytes prove the start dead.  Survivors go to the start queue (sqn = its fill level), which is run when full.
// TWO: the candidates are the byte pairs of the sweep filter (the two table steps still confirm each one).
template <int KIND, int NR, bool HIGH, bool TWO>
__device__ __noinline__ int sparse_run_units(const KParams& p, const SparseParams& sp, uint32_t s_table, uint32_t s_cmap,
                                             const SparseCtx& c, int count, int sqn) {
    const Table<KIND> T = sparse_table<KIND>(sp, s_table, s_cmap);
    const int lane = threadIdx.x & 31;
    const uint32_t FULL = 0xffffffffu;
    __syncwarp();
    uint32_t cand = 0, tile = 0, flag = 0;
    int64_t P = 0, t0 = 0;                                         // buffer position of the unit's byte 0; of the tile's
    if (lane < count) {
        const uint4 e = c.units[lane];
        tile = e.x; flag = e.y & 0x80000000u;
        const int64_t first = (int64_t)e.x * c.spt;
        const int cnt = (int)((c.n - first) < c.spt ? (c.n - first) : c.spt);
        t0 = sparse_off(c.offsets, c.stride, first);
        const int64_t tend = sparse_off(c.offsets, c.stride, first + cnt);
        const uintptr_t gbuf = reinterpret_cast<uintptr_t>(c.buf);
        const uintptr_t ua = ((gbuf + (uintptr_t)t0) & ~(uintptr_t)31) + ((((uintptr_t)e.w << 32) | e.z) << 5);
        const uint4 v0 = __ldg(reinterpret_cast<const uint4*>(ua)), v1 = __ldg(reinterpret_cast<const uint4*>(ua + 16));
        P = (int64_t)ua - (int64_t)gbuf;
        if (TWO) {
            // the byte after the unit, if it is in the tile; else a start on the unit's last byte is the last byte of
            // the tile's last string, and the byte is assumed to match
            const uint32_t sel = lead_sel(sp);
            uint32_t z_next = P + 32 < tend ? second_zero<true>(sp, __ldg(reinterpret_cast<const uint8_t*>(ua + 32)), sel) : 0u;
            const uint32_t w[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
            for (int k = 7; k >= 0; k--) {
                const uint32_t z = second_zero<true>(sp, w[k], sel);
                cand |= pack_byte_flags(pair_mask(sp, w[k], z, z_next) | (HIGH ? w[k] : 0u)) << (4 * k);
                z_next = z;
            }
        } else {
            cand = pack_byte_flags(first_mask<NR, HIGH>(sp, v0.x)) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v0.y)) << 4) |
                   (pack_byte_flags(first_mask<NR, HIGH>(sp, v0.z)) << 8) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v0.w)) << 12) |
                   (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.x)) << 16) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.y)) << 20) |
                   (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.z)) << 24) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.w)) << 28);
        }
        if (P < t0) cand &= 0xFFFFFFFFu << (int)(t0 - P);
        if (P + 32 > tend) cand &= (P >= tend) ? 0u : (0xFFFFFFFFu >> (int)(P + 32 - tend));
    }
    while (__any_sync(FULL, cand != 0)) {
        bool sv = false;
        int64_t pos = 0;
        if (cand) {
            pos = P + __ffs(cand) - 1;
            cand &= cand - 1;
            const uint32_t b = __ldg(c.buf + pos);
            const uint32_t w1 = T.next((uint32_t)sp.q0, b);
            if (w1 & (W_ACC | W_INTER)) sv = true;
            else if (w1 & W_STATE) {
                const uint32_t b1 = pos + 1 < c.total ? __ldg(c.buf + pos + 1) : 0u;      // may belong to the next string
                sv = ((T.next(w1, b1) | T.next(w1, 0u)) & (W_STATE | W_ACC)) != 0;
            }
        }
        const uint32_t m = __ballot_sync(FULL, sv);
        if (m) {
            const unsigned long long rel = (unsigned long long)(pos - t0);
            if (sv) c.starts[sqn + __popc(m & ((1u << lane) - 1))] = make_uint4(tile, SPARSE_START | flag, (uint32_t)rel, (uint32_t)(rel >> 32));
            sqn += __popc(m);
            if (sqn >= 32) {
                sparse_run_starts<KIND>(p, sp, s_table, s_cmap, c, 32);
                if (lane < sqn - 32) { const uint4 x = c.starts[32 + lane]; c.starts[lane] = x; }
                sqn -= 32;
                __syncwarp();
            }
        }
    }
    __syncwarp();
    return sqn;                                                    // the start queue's new fill level
}

// 4 CTAs per SM, 4 rows (4 KB per warp) in flight: the best of the measured combinations (DESIGN.md section 5)
static constexpr int SPARSE_CTAS_PER_SM = 4, SPARSE_ROWS = 4;

// One group of the sweep: rows r .. r + SPARSE_ROWS - 1 (32 units each) of a segment of `lim` units that starts at
// `sbase`.  Returns bit k set when this lane's unit in row r + k passed the filter.  WHOLE: every unit of the group lies
// in the segment, so nothing is bounds-tested or zeroed (all groups but a tile's last).
template <int NR, bool HIGH, bool TWO, bool WHOLE>
__device__ __forceinline__ uint32_t sweep_group(const SparseParams& sp, uintptr_t sbase, int r, int lim, uint32_t& seen) {
    const int lane = threadIdx.x & 31;
    uint4 va[SPARSE_ROWS], vb[SPARSE_ROWS];
#pragma unroll
    for (int k = 0; k < SPARSE_ROWS; k++) {            // all loads first: SPARSE_ROWS KB per warp in flight
        const int u = ((r + k) << 5) + lane;
        const uintptr_t a = sbase + ((uintptr_t)(uint32_t)u << 5);
        if (WHOLE || u < lim) {
            va[k] = ldg_nc_v4(reinterpret_cast<const void*>(a));
            vb[k] = ldg_nc_v4(reinterpret_cast<const void*>(a + 16));
        } else {
            va[k] = make_uint4(0, 0, 0, 0); vb[k] = va[k];
        }
    }
    // TWO: the first word of the next unit is in lane + 1 of the same row, or for lane 31 in lane 0 of the next row.
    // After the group's last row and after the segment's last unit the next unit is not loaded: it is assumed to match.
    uint32_t zn[SPARSE_ROWS];
    if (TWO) {
        const uint32_t sel = lead_sel(sp);
        uint32_t z0[SPARSE_ROWS];
#pragma unroll
        for (int k = 0; k < SPARSE_ROWS; k++) z0[k] = second_zero<true>(sp, va[k].x, sel);
#pragma unroll
        for (int k = 0; k < SPARSE_ROWS; k++) {
            const uint32_t give = lane != 0 ? z0[k] : k + 1 < SPARSE_ROWS ? z0[k + 1] : 0u;
            zn[k] = __shfl_sync(0xffffffffu, give, (lane + 1) & 31);
            if (!WHOLE && ((r + k) << 5) + lane + 1 >= lim) zn[k] = 0u;
        }
    }
    uint32_t bits = 0;
#pragma unroll
    for (int k = 0; k < SPARSE_ROWS; k++) {
        const int u = ((r + k) << 5) + lane;
        const uint32_t h = (WHOLE || u < lim) ? unit_any<NR, HIGH, TWO>(sp, va[k], vb[k], seen, TWO ? zn[k] : 0u) : 0u;
        bits |= (h ? 1u : 0u) << k;
    }
    return bits;
}

template <int KIND, int NR, bool HIGH, bool TWO>
__global__ void __launch_bounds__(256, SPARSE_CTAS_PER_SM) k_in_sparse(KParams p, SparseParams sp, const uint8_t* __restrict__ buf,
                                                                     const int64_t* __restrict__ offsets, int64_t n, int64_t total,
                                                                     uint8_t* __restrict__ out, int spt, int64_t ntiles,
                                                                     int table_smem_bytes, int prezeroed, int64_t stride) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_cmap = smem;
    uint8_t* s_table = smem + 256;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint4* s_units = reinterpret_cast<uint4*>(smem + sparse_shared_head(table_smem_bytes) + warp * SPARSE_WARP_BYTES);
    uint4* s_starts = s_units + 64;
    KParams anch = p;                       // stage_table reads table / classmap / sizes from a KParams
    anch.table = sp.table; anch.classmap = sp.classmap; anch.table_words = sp.table_words; anch.row_shift = sp.row_shift;
    Table<KIND> T = stage_table<KIND>(anch, s_table, s_cmap);
    // shared copies of the parameters for the out-of-line phases
    static_assert(sizeof(KParams) + sizeof(SparseParams) + 8 * sizeof(SparseCtx) <= SPARSE_PARAM_BYTES, "parameter block");
    uint8_t* s_params = smem + sparse_shared_head(table_smem_bytes) - SPARSE_PARAM_BYTES;
    KParams* sh_p = reinterpret_cast<KParams*>(s_params);
    SparseParams* sh_sp = reinterpret_cast<SparseParams*>(s_params + sizeof(KParams));
    SparseCtx* sh_c = reinterpret_cast<SparseCtx*>(s_params + sizeof(KParams) + sizeof(SparseParams)) + warp;
    if (threadIdx.x == 0) { *sh_p = p; *sh_sp = sp; }
    if (lane == 0) {
        sh_c->buf = buf; sh_c->offsets = offsets; sh_c->stride = stride; sh_c->out = out; sh_c->n = n; sh_c->total = total;
        sh_c->spt = spt;
        sh_c->units = s_units; sh_c->starts = s_starts;
    }
    __syncthreads();                        // the only block-wide step: table and parameter copies are staged
    const Anchored A{sp.flags, sp.start_nul, sp.q0};
    const uint32_t FULL = 0xffffffffu;
    const int nt = (int)ntiles;             // the host keeps n (hence ntiles) below 2^31

    // The warp's state machine.  The inner loop (no calls) advances it until 32 units or 32 starts are waiting or
    // the tiles are used up; the outer loop runs the queues and comes back.
    enum { ST_NEW = 0, ST_SWEEP = 1, ST_STRINGS = 2, ST_PUSH = 3 };
    int t = blockIdx.x * 8 + warp;          // tile in progress / next tile
    int st = ST_NEW, it = 0;                // it: next string (ST_STRINGS) or next row (ST_PUSH)
    int uqn = 0, sqn = 0;                   // queue fill levels (warp-uniform)
    int count = 0, nrows = 0;
    int64_t seg = 0, nunits = 0;            // rows [seg, seg + nrows) of the tile's units are being swept / pushed
    uintptr_t ubase = 0;                    // 32-byte aligned address of the tile's unit 0
    uint32_t hitbits = 0;                   // bit r: this lane's unit in row seg + r passed the filter
    bool high = false;
    int64_t nx0 = 0, nx1 = 0;               // byte range of the warp's next tile
    bool have_next = false;

    bool drain = false;                     // run the queues even if they are not full (the tiles are used up)
    for (;;) {
        for (;;) {
            if (uqn >= 32 || sqn >= 32 || drain) break;
            if (st == ST_NEW) {
                if (t >= nt) { drain = true; break; }
                const int64_t first = (int64_t)t * spt;
                count = (int)((n - first) < spt ? (n - first) : spt);
                const int64_t t0 = have_next ? nx0 : sparse_off(offsets, stride, first);
                const int64_t tend = have_next ? nx1 : sparse_off(offsets, stride, first + count);
                {   // the next tile's extents, asked for now, used when this tile is done
                    const int64_t fn = first + (int64_t)gridDim.x * 8 * spt;
                    have_next = fn < n;
                    if (have_next) { nx0 = sparse_off(offsets, stride, fn); nx1 = sparse_off(offsets, stride, fn + spt < n ? fn + spt : n); }
                }
                const uintptr_t g0 = reinterpret_cast<uintptr_t>(buf) + (uintptr_t)t0;
                ubase = g0 & ~(uintptr_t)31;
                nunits = tend > t0 ? (int64_t)((reinterpret_cast<uintptr_t>(buf) + (uintptr_t)tend - ubase + 31) >> 5) : 0;
                seg = 0;
                high = nunits > 1024;       // a tile swept in several segments: its winners are always re-checked
                st = ST_SWEEP;
            }
            if (st == ST_SWEEP) {
                // ---- S: up to 32 rows of 32 units, SPARSE_ROWS rows (SPARSE_ROWS KB per warp) in flight ----
                const int64_t left = nunits - seg;
                const int lim = (int)(left < 1024 ? left : 1024);  // units in this segment
                const uintptr_t sbase = ubase + ((uintptr_t)seg << 5);
                nrows = (lim + 31) >> 5;
                hitbits = 0;
                uint32_t seen = 0;
                int r = 0;
                for (; ((r + SPARSE_ROWS) << 5) <= lim; r += SPARSE_ROWS)
                    hitbits |= sweep_group<NR, HIGH, TWO, true>(sp, sbase, r, lim, seen) << r;
                if (r < nrows) hitbits |= sweep_group<NR, HIGH, TWO, false>(sp, sbase, r, lim, seen) << r;
                high = high || __any_sync(FULL, (seen & 0x80808080u) != 0);   // (bytes next to the tile are counted in: harmless)
                st = seg == 0 ? ST_STRINGS : ST_PUSH;              // the strings' own results are written before any unit is queued
                it = 0;
            }
            if (st == ST_STRINGS) {
                // ---- per string: degenerate texts, the start on the leading NUL ----
                const int64_t first = (int64_t)t * spt;
                if (prezeroed) it = count;                         // no string is decided here, and the host has cleared `out`
                while (it < count && sqn < 32) {
                    const int i = it + lane;
                    bool r = false, defer = false;
                    if (i < count) {
                        const int64_t o0 = sparse_off(offsets, stride, first + i), o1 = sparse_off(offsets, stride, first + i + 1);
                        const int64_t len = o1 - o0;
                        if (len == 0 || (len == 1 && __ldg(buf + o0) == 0x20)) r = p.q0_accepting != 0;   // api_internal_m.F90:68-74
                        else if (sp.start_nul != 0) {
                            r = attempt_wins(A, T, FetchGlobal{buf + o0}, len, (uint32_t)sp.start_nul, 0);
                            if (r && p.prefix_mode == 1 && high) { r = false; defer = true; }
                        }
                        out[first + i] = r ? 1 : 0;                // provisional for a deferred string
                    }
                    const uint32_t m = __ballot_sync(FULL, defer);
                    if (defer) s_starts[sqn + __popc(m & ((1u << lane) - 1))] = make_uint4((uint32_t)t, SPARSE_RECHECK, (uint32_t)i, 0u);
                    sqn += __popc(m);
                    it += 32;
                }
                if (it < count) continue;                          // queue full: run it, then resume here
                __syncwarp();                                      // results written before any start of this tile sets one
                st = ST_PUSH;
                it = 0;
            }
            // ---- queue the units that passed the filter ----
            while (it < nrows && uqn < 32) {
                const bool hit = (hitbits >> it) & 1u;
                const uint32_t m = __ballot_sync(FULL, hit);
                if (hit) {
                    const unsigned long long u = (unsigned long long)(seg + ((int64_t)it << 5) + lane);
                    s_units[uqn + __popc(m & ((1u << lane) - 1))] = make_uint4((uint32_t)t, high ? 0x80000000u : 0u, (uint32_t)u, (uint32_t)(u >> 32));
                }
                uqn += __popc(m);
                it++;
            }
            if (it < nrows) continue;                              // queue full: run it, then resume here
            seg += (int64_t)nrows << 5;
            if (seg < nunits) st = ST_SWEEP;
            else {
                // Tile finished.  Its queued units and starts stay in the queues and are run with the next tile's once
                // 32 are waiting; only after the warp's last tile are part-full queues drained.
                st = ST_NEW;
                t += gridDim.x * 8;
            }
        }
        // ---- outer loop: run a queue (the only calls of the kernel) ----
        if (uqn >= 32 || (drain && uqn > 0)) {
            const int run = uqn < 32 ? uqn : 32;
            sqn = sparse_run_units<KIND, NR, HIGH, TWO>(*sh_p, *sh_sp, T.s_table, T.s_cmap, *sh_c, run, sqn);
            if (lane < uqn - run) { const uint4 x = s_units[run + lane]; s_units[lane] = x; }
            uqn -= run;
            __syncwarp();
        } else if (sqn >= 32 || (drain && sqn > 0)) {
            const int run = sqn < 32 ? sqn : 32;
            sparse_run_starts<KIND>(*sh_p, *sh_sp, T.s_table, T.s_cmap, *sh_c, run);
            if (lane < sqn - run) { const uint4 x = s_starts[run + lane]; s_starts[lane] = x; }
            sqn -= run;
            __syncwarp();
        } else {
            drain = false;                                         // both queues are empty
            if (st == ST_NEW && t >= nt) break;                    // ... and no tiles are left
        }
    }
}

// K3: ragged batch, span result (config C3).  Same tiling as K2; the table words carry flag bits.
template <int KIND>
__global__ void __launch_bounds__(256) k_regex_ragged(KParams p, const uint8_t* __restrict__ buf,
                                                      const int64_t* __restrict__ offsets, int64_t n, int64_t total,
                                                      int64_t* __restrict__ from, int64_t* __restrict__ to,
                                                      int spt, int cap, int64_t ntiles, int table_smem_bytes) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_cmap = smem + 16;
    uint8_t* s_table = smem + 16 + 256;
    int32_t* s_off = reinterpret_cast<int32_t*>(smem + 16 + 256 + table_smem_bytes);
    uint8_t* tile = smem + tile_offset(table_smem_bytes, spt);
    const uint32_t mbar = smem_u32(smem);
    Table<KIND> T = stage_table<KIND>(p, s_table, s_cmap);
    if (threadIdx.x == 0) mbar_init(mbar, 1);
    __syncthreads();
    uint32_t phase = 0;
    const uint32_t tile_addr = smem_u32(tile);
    const bool plain = !p.all_active && !p.pre_active;   // brute-force starts, no literal machinery
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const TileCtx c = load_tile(buf, offsets, n, total, t, spt, cap, tile, s_off, mbar, phase);
        for (int i = threadIdx.x; i < c.count; i += blockDim.x) {
            const int32_t r0 = s_off[i], r1 = s_off[i + 1];
            int64_t f, e;
            if (r1 == OFF_BEYOND) {
                const int64_t o0 = __ldg(offsets + c.first + i), o1 = __ldg(offsets + c.first + i + 1);
                eval_regex(p, T, FetchGlobal{buf + o0}, o1 - o0, f, e);
            } else if (plain) {
                const int len = r1 - r0;
                const uint32_t a = tile_addr + (uint32_t)r0;
                f = 0; e = 0;
                if (!(len == 0 || (len == 1 && lds_u8(a) == 0x20))) {            // api_internal_m.F90:68-74
                    int64_t ff, tt;
                    brute_force_smem(Anchored{p.flags, p.start_nul, p.q0}, T, a, len, ff, tt);
                    if (ff > 0 && tt > 0) { f = ff; e = tt; }                        // forgex.F90:332-343
                }
            } else {
                eval_regex(p, T, FetchShared{tile_addr + (uint32_t)r0}, (int64_t)(r1 - r0), f, e);
            }
            from[c.first + i] = f;
            to[c.first + i] = e;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// K3f: ragged batch, span result, linear time (config C3).
// Forward: ONE walk of the "ordered groups" automaton (fx_automata.cpp, build_span_forward) yields the end of
// Forgex's leftmost-longest match: the last position at which the state held the exit.  Its table words carry every
// event of a step -- ACC (the new state holds the exit), RA (a broken multi-byte sequence replayed as U+FFFF bytes and
// passed an accept on the way; fx_internal.hpp W_RA) -- so a step is one lookup and, rarely, an update of `last`;
// the walker keeps no per-sequence bookkeeping.  Backward: the reverse automaton (over code-point classes) walks from
// that end towards the front, decoding characters backwards with the reference's decoder rule (a well-formed sequence
// that ends exactly here, else one byte = U+FFFF); the class of a character comes from a two-level table in shared
// memory, the transition word carries "this state holds the NFA entry"; the leftmost such position is the start.
// ---------------------------------------------------------------------------------------------
static constexpr uint32_t W_SSTATE = 0x0FFFu, W_RA = 0x3000u;
static constexpr int SPAN_ROW = 258;             // u16 entries per state row in shared memory: 129 words, an odd stride, so that
                                                 // lanes in different states reading the same byte value hit different banks
struct SpanParams {
    // forward automaton (span words)
    const uint16_t* direct;     // nstates x 256
    const uint16_t* table;      // class-compressed: nstates << row_shift
    const uint8_t* classmap;
    const uint8_t* endinfo;     // nstates
    int nstates, row_shift, start, start_acc;
    // reverse automaton over code-point classes
    const uint16_t* rdelta;     // rstates x rclasses, bit 15 = the destination holds the NFA entry
    const uint8_t* rpage;       // 1024 (nullptr: no two-level map, binary search)
    const uint8_t* rmixed;
    const int32_t* cuts;        // rclasses + 1 ascending code points
    int rstates, rclasses, rstart, nul_class, ffff_class, nmixed;
};

// forward table access.  FK 0: 256 columns, padded rows, shared memory; FK 1: class-compressed, shared; FK 2: class-compressed, global
template <int FK>
struct SpanFwd {
    uint32_t s_table, s_cmap;
    const uint16_t* g_table;
    const uint8_t* g_cmap;
    int shift;
    __device__ __forceinline__ uint32_t next(uint32_t st, uint32_t b) const {
        if (FK == 0) return lds_u16(s_table + st * (SPAN_ROW * 2) + b * 2);
        if (FK == 1) return lds_u16(s_table + (((st << shift) + lds_u8(s_cmap + b)) << 1));
        return __ldg(g_table + ((st << shift) + __ldg(g_cmap + b)));
    }
};
// reverse tables.  RS true: rdelta / page / mixed in shared memory
template <bool RS>
struct SpanRev {
    uint32_t s_delta, s_page, s_mixed;
    __device__ __forceinline__ uint32_t delta(const SpanParams& sp, uint32_t r, uint32_t c) const {
        if (RS) return lds_u16(s_delta + ((r * (uint32_t)sp.rclasses + c) << 1));
        return __ldg(sp.rdelta + r * (uint32_t)sp.rclasses + c);
    }
    __device__ __forceinline__ uint32_t cls(const SpanParams& sp, uint32_t cp) const {
        if (cp < 0x10000u && sp.rpage != nullptr) {
            const uint32_t pg = RS ? lds_u8(s_page + (cp >> 6)) : (uint32_t)__ldg(sp.rpage + (cp >> 6));
            if (pg < 0x80u) return pg;
            const uint32_t i = ((pg & 0x7Fu) << 6) | (cp & 63u);
            return RS ? lds_u8(s_mixed + i) : (uint32_t)__ldg(sp.rmixed + i);
        }
        int lo = 0, hi = sp.rclasses;              // largest c with cuts[c] <= cp
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if ((uint32_t)__ldg(sp.cuts + mid) <= cp) lo = mid; else hi = mid;
        }
        return (uint32_t)lo;
    }
};

// one forward step: the byte at text index jj
#define FX_SPAN_STEP(T, st, last, b, jj)                                         \
    {                                                                             \
        const uint32_t nw_ = (T).next((st), (b));                                 \
        if (nw_ & 0xB000u) {                                                      \
            if (nw_ & W_RA) (last) = (jj) + 1 - (int)((nw_ >> 12) & 3u);          \
            if (nw_ & W_ACC) (last) = (jj) + 1;                                   \
        }                                                                         \
        (st) = nw_ & W_SSTATE;                                                    \
    }

// The books of four transition words that have already been looked up (the deferred-flag loops: four lookups, one OR
// test).  A step's event ASSIGNS `last` (an accept: the position behind the byte; a replay mark: 1..3 bytes before
// that), so of the four steps only the last one that holds an event counts -- picked with selects, no second walk.
// (On C3 some lane of a warp sees an event in nearly every word -- seven accepts in a row per \w{2,8} -- so this runs
// almost every iteration: it has to be short.)
#define FX_SPAN_BOOKS4(n1, n2, n3, n4, last, jj)                                  \
    {                                                                             \
        uint32_t ev_ = (n1);                                                      \
        int k_ = 1;                                                               \
        if ((n2) & 0xB000u) { ev_ = (n2); k_ = 2; }                               \
        if ((n3) & 0xB000u) { ev_ = (n3); k_ = 3; }                               \
        if ((n4) & 0xB000u) { ev_ = (n4); k_ = 4; }                               \
        if (ev_ & 0xB000u) (last) = (jj) + k_ - ((ev_ & W_ACC) ? 0 : (int)((ev_ >> 12) & 3u)); \
    }

// what the end of the text does in state st (the pending bytes of an unfinished sequence replay as U+FFFF; the
// trailing NUL is consumed but is not a start)
__device__ __forceinline__ int span_end_of_text(const SpanParams& sp, uint32_t st, int len, int last) {
    const uint32_t e = __ldg(sp.endinfo + st);
    if (e & 3u) last = len + 1 - (int)(e & 3u);
    if (e & 4u) last = len + 1;
    return last;
}

// backward half: the leftmost start of a match that ends at `last` (> 0).  Returns from (1-based), 0 if none.
template <bool RS, class FETCH>
__device__ __forceinline__ int span_backward(const SpanParams& sp, const SpanRev<RS>& R, FETCH fetch, int len, int last) {
    uint32_t r = (uint32_t)sp.rstart;
    int pos = last;
    if (last > len) { r = R.delta(sp, r, (uint32_t)sp.nul_class) & 0x7FFFu; pos = len; }
    int best = -2;                                          // -2 none, -1 the leading NUL, >= 0 text index
    while (r != 0 && pos > 0) {
        uint32_t c = fetch(pos - 1);                        // the character that ends at pos
        int q = pos - 1;
        uint32_t cp = c;
        if (c >= 0x80u) {
            cp = 0xFFFFu;                                   // stray / malformed byte unless a well-formed sequence ends here
            if ((c & 0xC0u) == 0x80u && pos >= 2) {
                const uint32_t d1 = fetch(pos - 2);
                if ((d1 & 0xE0u) == 0xC0u) { cp = ((d1 & 0x1Fu) << 6) | (c & 0x3Fu); q = pos - 2; }
                else if ((d1 & 0xC0u) == 0x80u && pos >= 3) {
                    const uint32_t d2 = fetch(pos - 3);
                    if ((d2 & 0xF0u) == 0xE0u) { cp = ((d2 & 0x0Fu) << 12) | ((d1 & 0x3Fu) << 6) | (c & 0x3Fu); q = pos - 3; }
                    else if ((d2 & 0xC0u) == 0x80u && pos >= 4) {
                        const uint32_t d3 = fetch(pos - 4);
                        if ((d3 & 0xF8u) == 0xF0u) {
                            cp = ((d3 & 0x07u) << 18) | ((d2 & 0x3Fu) << 12) | ((d1 & 0x3Fu) << 6) | (c & 0x3Fu);
                            q = pos - 4;
                        }
                    }
                }
            }
        }
        const uint32_t w = R.delta(sp, r, R.cls(sp, cp));
        r = w & 0x7FFFu;
        if (r == 0) break;
        pos = q;
        if (w & 0x8000u) best = pos;
    }
    if (r != 0 && pos == 0) {                               // the leading NUL sentinel (start position 1)
        const uint32_t w = R.delta(sp, r, (uint32_t)sp.nul_class);
        if ((w & 0x7FFFu) != 0 && (w & 0x8000u)) best = -1;
    }
    if (best == -2) return 0;                               // cannot happen for a consistent pair of automata
    return best < 0 ? 1 : best + 1;
}

// the linear-time span search over any byte source (strings that are not staged: longer than a warp's tile)
template <int FK, bool RS, class FETCH>
__device__ __noinline__ void span_linear(const SpanParams& sp, const SpanFwd<FK>& T, const SpanRev<RS>& R, FETCH fetch, int len,
                                         int64_t& from, int64_t& to) {
    from = 0; to = 0;
    uint32_t st = (uint32_t)sp.start;
    int last = sp.start_acc ? 0 : -1;
    int j = 0;
    for (; j < len && st != 0; j++) { const uint32_t b = fetch(j); FX_SPAN_STEP(T, st, last, b, j); }
    if (st != 0) last = span_end_of_text(sp, st, len, last);
    if (last <= 0) return;                                  // no match, or only the leading NUL matched (to = 0)
    const int f = span_backward(sp, R, fetch, len, last);
    if (f > 0) { from = f; to = last < len ? last : len; }
}

// shared memory of K3f: classmap 256 | forward table | reverse tables (delta, page 1024, mixed) | pad to 128 |
//   SPAN_WARPS warp regions of `warp_bytes`:
//   [0,16) mbarrier | offsets (spt+4) x int32 | results spt x int2 | queue spt x uint32 | claim order spt x uint16 |
//   32 bucket counters | pad to 128 | tile (cap + 64)
// Every warp stages its own tiles (its own TMA bulk copy on its own mbarrier): no block-wide step after the tables are
// staged.  One CTA of 32 warps per SM: one copy of the tables, the rest of the shared memory is tile space.
static constexpr int SPAN_WARPS = 32;
struct SpanLayout { int off_res, off_queue, off_perm, off_hist, off_tile, warp_bytes; };
__host__ __device__ __forceinline__ SpanLayout span_layout(int spt, int cap) {
    SpanLayout L;
    L.off_res = (16 + (spt + 4) * 4 + 7) & ~7;          // int2 entries
    L.off_queue = L.off_res + spt * 8;
    L.off_perm = L.off_queue + spt * 4;
    L.off_hist = (L.off_perm + spt * 2 + 3) & ~3;
    L.off_tile = (L.off_hist + 128 + 127) & ~127;
    L.warp_bytes = (L.off_tile + cap + 64 + 127) & ~127;
    return L;
}
struct SpanHead { int off_rdelta, off_page, off_mixed, bytes; };
__host__ __device__ __forceinline__ SpanHead span_head(int fwd_bytes, int rdelta_bytes, int nmixed, bool rs) {
    SpanHead H;
    H.off_rdelta = (256 + fwd_bytes + 15) & ~15;
    H.off_page = H.off_rdelta + (rs ? ((rdelta_bytes + 15) & ~15) : 0);
    H.off_mixed = H.off_page + (rs ? 1024 : 0);
    H.bytes = (H.off_mixed + (rs ? nmixed * 64 : 0) + 127) & ~127;
    return H;
}
static constexpr int SPAN_ROUND = 64;            // bytes a lane walks before the warp looks for idle lanes again (C3: 16 -> 701, 32 -> 777, 64 -> 816 GB/s)

template <int FK, bool RS>
__global__ void __launch_bounds__(SPAN_WARPS * 32, 1) k_span_ragged(KParams p, SpanParams sp, const uint8_t* __restrict__ buf,
                                                                        const int64_t* __restrict__ offsets, int64_t n, int64_t total,
                                                                        int64_t* __restrict__ from, int64_t* __restrict__ to,
                                                                        int spt, int cap, int64_t ntiles, int fwd_bytes) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t FULL = 0xffffffffu;
    const SpanHead H = span_head(fwd_bytes, sp.rstates * sp.rclasses * 2, sp.nmixed, RS);
    const SpanLayout L = span_layout(spt, cap);
    // ---- stage the tables (the only block-wide step) ----
    SpanFwd<FK> T;
    T.s_cmap = smem_u32(smem); T.s_table = smem_u32(smem + 256); T.g_table = sp.table; T.g_cmap = sp.classmap; T.shift = sp.row_shift;
    if (FK == 0) {                                           // rows of 256 entries -> rows of SPAN_ROW entries
        uint16_t* dst = reinterpret_cast<uint16_t*>(smem + 256);
        for (int i = threadIdx.x; i < sp.nstates * 128; i += blockDim.x) {
            const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(sp.direct) + i);
            const int st = i >> 7, c = (i & 127) << 1;
            *reinterpret_cast<uint32_t*>(dst + st * SPAN_ROW + c) = v;
        }
    } else if (FK == 1) {
        uint32_t* dst = reinterpret_cast<uint32_t*>(smem + 256);
        const int words32 = ((sp.nstates << sp.row_shift) + 1) >> 1;
        for (int i = threadIdx.x; i < words32; i += blockDim.x) dst[i] = __ldg(reinterpret_cast<const uint32_t*>(sp.table) + i);
        for (int i = threadIdx.x; i < 64; i += blockDim.x)
            reinterpret_cast<uint32_t*>(smem)[i] = __ldg(reinterpret_cast<const uint32_t*>(sp.classmap) + i);
    }
    SpanRev<RS> R;
    R.s_delta = smem_u32(smem + H.off_rdelta); R.s_page = smem_u32(smem + H.off_page); R.s_mixed = smem_u32(smem + H.off_mixed);
    if (RS) {
        uint16_t* d = reinterpret_cast<uint16_t*>(smem + H.off_rdelta);
        for (int i = threadIdx.x; i < sp.rstates * sp.rclasses; i += blockDim.x) d[i] = __ldg(sp.rdelta + i);
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) smem[H.off_page + i] = __ldg(sp.rpage + i);
        for (int i = threadIdx.x; i < sp.nmixed * 64; i += blockDim.x) smem[H.off_mixed + i] = __ldg(sp.rmixed + i);
    }
    uint8_t* region = smem + H.bytes + warp * L.warp_bytes;
    int32_t* s_off = reinterpret_cast<int32_t*>(region + 16);
    int2* s_res = reinterpret_cast<int2*>(region + L.off_res);
    uint32_t* s_queue = reinterpret_cast<uint32_t*>(region + L.off_queue);
    uint16_t* s_perm = reinterpret_cast<uint16_t*>(region + L.off_perm);
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(region + L.off_hist);
    uint8_t* tile = region + L.off_tile;
    const uint32_t mbar = smem_u32(region);
    if (lane == 0) mbar_init(mbar, 1);
    __syncthreads();
    uint32_t phase = 0;
    const uint32_t tile_addr = smem_u32(tile);
    const uintptr_t gbuf = reinterpret_cast<uintptr_t>(buf);
    const int64_t nwarps = (int64_t)gridDim.x * SPAN_WARPS;
    for (int64_t t = (int64_t)blockIdx.x * SPAN_WARPS + warp; t < ntiles; t += nwarps) {
        // ---- stage the tile: strings [first, first + count), up to `cap` bytes of them ----
        const int64_t first = t * spt;
        const int count = (int)((n - first) < spt ? (n - first) : spt);
        const int64_t t0 = __ldg(offsets + first), tend = __ldg(offsets + first + count);
        const int64_t t1 = tend - t0 > cap ? t0 + cap : tend;
        const uintptr_t g0 = gbuf + (uintptr_t)t0;
        const int64_t base = t0 - (int64_t)(g0 & 15);              // tile[0] = byte `base` (the bulk source is 16-byte aligned)
        const uintptr_t gsrc = g0 & ~(uintptr_t)15;
        uintptr_t gcopy_end = (gbuf + (uintptr_t)t1 + 15) & ~(uintptr_t)15;
        const uintptr_t gsafe_end = (gbuf + (uintptr_t)total) & ~(uintptr_t)15;   // never bulk-read past the last whole 16-byte block
        if (gcopy_end > gsafe_end) gcopy_end = gsafe_end;
        const uint32_t bulk = gcopy_end > gsrc ? (uint32_t)(gcopy_end - gsrc) : 0u;
        __syncwarp();                                              // every lane is done with the previous tile
        if (bulk && lane == 0) {
            mbar_expect_tx(mbar, bulk);
            bulk_g2s(tile_addr, reinterpret_cast<const void*>(gsrc), bulk, mbar);
        }
        for (int64_t x = (int64_t)(gsrc + bulk) - (int64_t)gbuf + lane; x < t1; x += 32)   // < 16 bytes at the very end of the buffer
            if (x >= t0) tile[x - base] = __ldg(buf + x);
        for (int i = lane; i <= count; i += 32) {                  // overlaps with the bulk copy in flight
            const int64_t o = __ldg(offsets + first + i);
            s_off[i] = o > t1 ? OFF_BEYOND : (int32_t)(o - base);
        }
        // ---- claim order: the longest strings first (counting sort over 8-byte length buckets; also while the copy is in
        // flight).  A tile gives a lane one or two strings; claimed in text order, the warp then waits for whichever lane
        // drew a long string last -- with the long ones out first the short ones fill the gaps (46 % -> 58 % busy lanes
        // on C3 at 45 strings per tile).  The results do not depend on the order.
        const bool ordered = count > 32;
        if (ordered) {
            s_hist[lane] = 0;
            __syncwarp();
            for (int i = lane; i < count; i += 32) {
                const int32_t r0 = s_off[i], r1 = s_off[i + 1];
                const int b = r1 == OFF_BEYOND ? 0 : 31 - (((r1 - r0) >> 3) < 31 ? ((r1 - r0) >> 3) : 31);   // bucket 0 = longest
                atomicAdd(s_hist + b, 1u);
            }
            __syncwarp();
            const uint32_t h = s_hist[lane];
            uint32_t x = h;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(FULL, x, d); if (lane >= d) x += y; }
            __syncwarp();
            s_hist[lane] = x - h;
            __syncwarp();
            for (int i = lane; i < count; i += 32) {
                const int32_t r0 = s_off[i], r1 = s_off[i + 1];
                const int b = r1 == OFF_BEYOND ? 0 : 31 - (((r1 - r0) >> 3) < 31 ? ((r1 - r0) >> 3) : 31);
                s_perm[atomicAdd(s_hist + b, 1u)] = (uint16_t)i;
            }
        }
        if (bulk) { mbar_wait(mbar, phase); phase ^= 1; }
        __syncwarp();
        // ---- forward walks.  The lanes are a pool of walkers: a lane that has no string claims the tile's next one;
        // all lanes then walk up to SPAN_ROUND bytes (whole 32-bit words of the tile) and the warp looks again.  A string
        // whose walk ends with a match is queued for the backward phase; the others get (0, 0).
        int next = 0, nq = 0;                                      // warp-uniform: next unclaimed string, queue fill
        bool have = false;
        int sidx = 0, len = 0, j = 0, last = -1;
        uint32_t a = 0, st = 0;
        for (;;) {
            const uint32_t idle = __ballot_sync(FULL, !have);
            if (idle) {
                const int mine = next + __popc(idle & ((1u << lane) - 1));
                if (!have && mine < count) {
                    sidx = ordered ? (int)s_perm[mine] : mine;
                    const int32_t r0 = s_off[sidx], r1 = s_off[sidx + 1];
                    if (r1 == OFF_BEYOND) {      // not staged (longer than a warp's tile): the same two walks, text from global memory
                        const int64_t o0 = __ldg(offsets + first + sidx), o1 = __ldg(offsets + first + sidx + 1);
                        int64_t f = 0, e = 0;
                        if (o1 - o0 == 0 || (o1 - o0 == 1 && __ldg(buf + o0) == 0x20)) {
                            // api_internal_m.F90:68-74: empty text or a lone blank never reaches the loop -> (0, 0)
                        } else if (o1 - o0 < 0x7FFFFFF0ll) {
                            span_linear(sp, T, R, FetchGlobal{buf + o0}, (int)(o1 - o0), f, e);
                        } else {                 // 2 GiB and more in one string: 64-bit positions, the anchored emulation
                            Table<3> G;
                            G.g_table = p.ctable; G.g_cmap = p.classmap; G.shift = p.c_row_shift; G.s_table = 0; G.s_cmap = 0;
                            eval_regex(p, G, FetchGlobal{buf + o0}, o1 - o0, f, e);
                        }
                        from[first + sidx] = f; to[first + sidx] = e;
                        s_res[sidx] = make_int2(-1, -1);           // already written
                    } else {
                        len = r1 - r0;
                        a = tile_addr + (uint32_t)r0;
                        if (len == 0 || (len == 1 && lds_u8(a) == 0x20)) s_res[sidx] = make_int2(0, 0);   // api_internal_m.F90:68-74
                        else { have = true; j = 0; st = (uint32_t)sp.start; last = sp.start_acc ? 0 : -1; }
                    }
                }
                next += __popc(idle);
                if (next > count) next = count;
            }
            if (!__any_sync(FULL, have)) { if (next >= count) break; else continue; }
            if (have) {
                int jend = (int)(((a + (uint32_t)j + SPAN_ROUND) & ~3u) - a);     // the round ends on a word boundary of the tile
                if (jend > len) jend = len;
                while (j < jend && ((a + (uint32_t)j) & 3u)) { const uint32_t b = lds_u8(a + j); FX_SPAN_STEP(T, st, last, b, j); j++; }
                for (; j + 4 <= jend && st != 0; j += 4) {
                    // four steps without looking at the flag bits; only a word that held an event (accept, replay mark:
                    // rare) is walked again with the books
                    const uint32_t w4 = lds_u32(a + j);
                    const uint32_t n1 = T.next(st, w4 & 0xFFu);
                    const uint32_t n2 = T.next(n1 & W_SSTATE, (w4 >> 8) & 0xFFu);
                    const uint32_t n3 = T.next(n2 & W_SSTATE, (w4 >> 16) & 0xFFu);
                    const uint32_t n4 = T.next(n3 & W_SSTATE, w4 >> 24);
                    if ((n1 | n2 | n3 | n4) & 0xB000u) {
                        FX_SPAN_BOOKS4(n1, n2, n3, n4, last, j);
                    }
                    st = n4 & W_SSTATE;
                }
                if (st != 0) for (; j < jend; j++) { const uint32_t b = lds_u8(a + j); FX_SPAN_STEP(T, st, last, b, j); }
                if (st == 0 || j >= len) {                          // this walk is over
                    if (st != 0) last = span_end_of_text(sp, st, len, last);
                    have = false;
                    if (last <= 0) s_res[sidx] = make_int2(0, 0);   // no match, or only the leading NUL matched (to = 0)
                }
            }
            // queue the strings whose walk ended with a match
            const bool push = !have && last > 0;
            const uint32_t pm = __ballot_sync(FULL, push);
            if (push) { s_queue[nq + __popc(pm & ((1u << lane) - 1))] = ((uint32_t)sidx << 16) | (uint32_t)last; last = -1; }
            nq += __popc(pm);
        }
        __syncwarp();
        // ---- backward walks, 32 queued strings at a time ----
        for (int q0 = 0; q0 < nq; q0 += 32) {
            if (q0 + lane < nq) {
                const uint32_t e = s_queue[q0 + lane];
                const int si = (int)(e >> 16), lst = (int)(e & 0xFFFFu);
                const int32_t r0 = s_off[si];
                const int ln = s_off[si + 1] - r0;
                const int f = span_backward(sp, R, FetchShared{tile_addr + (uint32_t)r0}, ln, lst);
                s_res[si] = f > 0 ? make_int2(f, lst < ln ? lst : ln) : make_int2(0, 0);
            }
        }
        __syncwarp();
        // ---- results, coalesced ----
        for (int i = lane; i < count; i += 32) {
            const int2 r = s_res[i];
            if (r.x >= 0) { from[first + i] = r.x; to[first + i] = r.y; }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K4: one long buffer, span result (config C4).
// The reference tries every character boundary as a start, in order, and returns at the first one
// whose anchored run accepts after >= 1 symbol (api_internal_m.F90:108-155).  The attempts are
// independent of each other, so they run in parallel: every thread takes 16 consecutive start
// candidates out of a coalesced 16-byte load, filters them with the first transition out of q0,
// and runs the surviving attempts forward through global memory.  The smallest winning start is
// kept with a 64-bit atomicMin; a second tiny kernel re-runs that one attempt to get the longest
// end.  Blocks sweep the buffer front to back and stop once their region lies behind the best
// start found so far.
// ---------------------------------------------------------------------------------------------
static constexpr unsigned long long NO_START = ~0ull;

// is text index pos a character boundary of the sequential strict decoder?  (pos holds a 10xxxxxx byte)
__device__ inline bool continuation_is_boundary(const uint8_t* __restrict__ s, int64_t len, int64_t pos) {
    for (int back = 1; back <= 3; back++) {
        const int64_t q = pos - back;
        if (q < 0) return true;
        const uint32_t b = __ldg(s + q);
        if ((b & 0xC0) == 0x80) continue;            // still inside a run of continuation bytes
        int n = (b >> 5) == 6 ? 2 : (b >> 4) == 14 ? 3 : (b >> 3) == 30 ? 4 : 1;
        if (n <= back) return true;                  // the sequence that starts at q ends before pos
        if (q + n > len) return true;                // truncated sequence: every byte stands alone
        for (int k = 1; k < n; k++)
            if ((__ldg(s + q + k) & 0xC0) != 0x80) return true;   // malformed: every byte stands alone
        return false;                                // pos is inside a well-formed sequence
    }
    return true;                                     // three continuation bytes in front: pos cannot be covered
}

// One candidate start (text index pos, first byte b): boundary check, then the anchored attempt, reading the text
// from global memory.  `open_end`: the window is followed by more text that this GPU does not hold; an attempt
// that is still alive at the window end cannot be decided here and is reported through *overflow.
// Work budget of a scan (K4): the attempts count their byte steps; when their sum passes `limit` the scan gives up
// (*abort = 1, every warp leaves) and the linear-time state-map scan (K5) answers instead.  limit == 0: no budget.
struct ScanBudget {
    unsigned long long* work;    // steps so far (all warps)
    unsigned long long* abort;   // set once the budget is spent
    unsigned long long limit;
};
static constexpr int BUDGET_TICK = 65536;        // steps a lane walks between two looks at the shared counter (one atomic each:
                                                 // at 4096 the 420 K same-address atomics of C4's attempts cost 3 ms of its 15)
__device__ __forceinline__ bool budget_spent(const ScanBudget& B, unsigned long long steps) {
    if (B.limit == 0) return false;
    const unsigned long long before = atomicAdd(B.work, steps);
    if (before + steps > B.limit) { *reinterpret_cast<volatile unsigned long long*>(B.abort) = 1ull; return true; }
    return *reinterpret_cast<volatile unsigned long long*>(B.abort) != 0;
}

// The part of an anchored attempt behind its plain stretch: from state `st` in front of text index `at` (no accept seen
// so far) with the full bookkeeping of run_attempt -- accepts, multi-byte sequences and their U+FFFF replay, the
// virtual trailing NUL.  `open_end`: the window is followed by text this GPU does not hold; an attempt that reaches the
// window end alive and without an accept cannot be decided here (*overflow).  Budgeted scans tick here as well.
template <int KIND>
__device__ __forceinline__ bool attempt_tail(const KParams& p, const Table<KIND>& T, const uint8_t* __restrict__ buf, int64_t len,
                                          uint32_t st, int64_t at, bool open_end, unsigned long long* overflow, const ScanBudget& B) {
    uint32_t w = st;
    int64_t seq = 0, last = -1;
    bool inter = false;
    for (int64_t j = at; j <= len; j++) {
        if (B.limit != 0 && ((j - at) & (BUDGET_TICK - 1)) == BUDGET_TICK - 1 && budget_spent(B, BUDGET_TICK)) return false;
        if (j == len && open_end) { if (last >= 0) return true; atomicAdd(overflow, 1ull); return false; }
        const uint32_t c = j < len ? __ldg(buf + j) : 0u;            // virtual trailing NUL at j == len
        if (inter && (c & 0xC0) != 0x80) {                            // sequence broken: pending bytes replay as U+FFFF
            const uint32_t f = __ldg(p.flags + (w & W_STATE));
            for (int k = 1; k <= (int)(j - seq); k++) if (f & (SF_FAILACC1 << (k - 1))) last = seq + k;
            inter = false;
        }
        const uint32_t nw = T.next(w & W_STATE, c);
        if ((nw & W_INTER) && !inter) seq = j;
        inter = (nw & W_INTER) != 0;
        w = nw;
        if (w & W_ACC) last = j + 1;
        if ((w & W_STATE) == 0) break;
    }
    return last >= 0;
}

template <int KIND>
__device__ __forceinline__ bool try_start(const KParams& p, const Table<KIND>& T, const uint8_t* __restrict__ buf,
                                          int64_t len, int64_t pos, uint32_t b, bool open_end,
                                          unsigned long long* overflow, const ScanBudget& B, uint32_t& acc) {
    if ((b & 0xC0) == 0x80 && !continuation_is_boundary(buf, len, pos)) return false;
    // The plain stretch first: as long as the next state neither accepts nor enters a multi-byte sequence, a step is
    // one load and one lookup (for C4 that is the whole line behind `^ERROR`).  Whatever comes then goes through the
    // general loop, from the state and position reached (no accept has been seen so far).
    uint32_t st = (uint32_t)p.q0;
    int64_t at = pos;
    for (;;) {
        int64_t stop = at + BUDGET_TICK < len ? at + BUDGET_TICK : len;
        const int64_t from = at;
        bool out = false;
        while (at < stop) {
            const uint32_t nw = T.next(st, __ldg(buf + at));
            if (nw & (W_ACC | W_INTER)) { out = true; break; }
            if (nw == 0) { acc += (uint32_t)(at - from); return false; }
            st = nw;
            at++;
        }
        acc += (uint32_t)(at - from);
        if (acc >= BUDGET_TICK) { const uint32_t a = acc; acc = 0; if (budget_spent(B, a)) return false; }
        if (out || at >= len) break;
    }
    return attempt_tail(p, T, buf, len, st, at, open_end, overflow, B);
}

// K4 window description: the kernel scans starts [start_lo, start_hi) of a window of `len` bytes that is a piece of
// a longer text; `origin` = text position of window byte 0 (keys written to `best` are global S positions).
struct ScanWindow {
    int64_t len, start_lo, start_hi, origin;
    int first;   // window begins at the true start of the text (the leading-NUL start belongs to it)
    int last;    // window ends at the true end of the text (the trailing NUL follows it)
};

// shared-memory layout of K4: classmap 256 | table | first-byte filter 256 | per-warp queues 8 x 64 x int64
__host__ __device__ __forceinline__ int scan_smem_bytes(int table_smem_bytes) {
    return 256 + table_smem_bytes + 256 + 8 * 64 * 8;
}

// Filter + attempts in one sweep, organised per warp.  A warp takes 32 consecutive 16-byte units with one
// coalesced load (each lane = 16 candidate starts).  First-byte filter: one shared-memory byte per candidate.
// Second-byte filter: drop a start when two bytes already prove it dead.  Survivors are compacted into a
// warp-private queue; whenever 32 are waiting, the 32 lanes run 32 attempts side by side (reading the text
// through L1/L2), so the rare long attempts never leave 31 lanes idle.
template <int KIND>
__global__ void __launch_bounds__(256) k_buffer_scan(KParams p, const uint8_t* __restrict__ buf, ScanWindow W,
                                                     unsigned long long* __restrict__ best, int table_smem_bytes,
                                                     const unsigned long long* __restrict__ gate,
                                                     const unsigned long long* __restrict__ run_if) {
    if (gate != nullptr && *gate != 0) return;      // the prefix occurs in the text: its occurrences were the candidates
    if (run_if != nullptr && *run_if == 0) return;  // fallback behind the state-map scan: only if that scan declined
    const ScanBudget B{nullptr, nullptr, 0ull};
    uint32_t acc = 0;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_cmap = smem;
    uint8_t* s_table = smem + 256;
    uint8_t* s_first = smem + 256 + table_smem_bytes;   // does byte b survive the step out of q0?
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t* queue = reinterpret_cast<int64_t*>(smem + 256 + table_smem_bytes + 256) + warp * 64;
    Table<KIND> T = stage_table<KIND>(p, s_table, s_cmap);
    __syncthreads();
    const uint32_t q0 = (uint32_t)p.q0;
    for (int b = threadIdx.x; b < 256; b += blockDim.x) s_first[b] = (T.next(q0, (uint32_t)b) & W_STATE) != 0;
    __syncthreads();
    const uint32_t first_addr = smem_u32(s_first);
    const int64_t len = W.len;
    const bool open_end = !W.last;
    unsigned long long* overflow = best + 1;
    const uint32_t FULL = 0xffffffffu;
    if (blockIdx.x == 0 && threadIdx.x == 0 && W.first) {   // start 1 = the leading NUL sentinel
        const Anchored A{p.flags, p.start_nul, p.q0};
        if (attempt_at(A, T, FetchGlobal{buf}, len, 1) >= 0) atomicMin(best, 1ull);
    }
    // 16-byte units aligned to the buffer ADDRESS; the unaligned head and the tail go through the same filter
    // one byte at a time (warp 0 of block 0 / last block)
    const uintptr_t g = reinterpret_cast<uintptr_t>(buf) + (uintptr_t)W.start_lo;
    int64_t head = W.start_lo + (int64_t)((16 - (g & 15)) & 15);
    if (head > W.start_hi) head = W.start_hi;
    const int64_t nvec = (W.start_hi - head) >> 4;
    const int64_t tail = head + (nvec << 4);
    int qn = 0;   // warp-uniform queue fill

    auto run_batch = [&](int count) {
        __syncwarp();
        if (lane < count) {
            const int64_t pos = queue[lane];
            if (try_start(p, T, buf, len, pos, __ldg(buf + pos), open_end, overflow, B, acc))
                atomicMin(best, (unsigned long long)(W.origin + pos) + 2);
        }
        __syncwarp();
    };
    auto push = [&](bool survive, int64_t pos) {
        const uint32_t m = __ballot_sync(FULL, survive);
        if (survive) queue[qn + __popc(m & ((1u << lane) - 1))] = pos;
        qn += __popc(m);
        if (qn >= 32) {
            run_batch(32);
            if (lane < qn - 32) { const int64_t v = queue[32 + lane]; queue[lane] = v; }
            qn -= 32;
            __syncwarp();
        }
    };
    auto second_byte_ok = [&](uint32_t b, uint32_t b1) -> bool {
        // keep the start unless two bytes prove it dead; undecidable (keep) when the first step accepts or enters a
        // multi-byte sequence (a broken sequence replays as U+FFFF and may accept on the way)
        const uint32_t w1 = T.next(q0, b);
        if (w1 & (W_ACC | W_INTER)) return true;
        const uint32_t w2 = T.next(w1 & W_STATE, b1);
        return (w2 & (W_STATE | W_ACC)) != 0;
    };

    const int64_t gwarp = (int64_t)blockIdx.x * 8 + warp, nwarps = (int64_t)gridDim.x * 8;
    if (gwarp == 0) {   // head and tail bytes, 32 at a time
        for (int64_t base = W.start_lo; base < head; base += 32) {
            const int64_t pos = base + lane;
            bool sv = false;
            if (pos < head) {
                const uint32_t b = __ldg(buf + pos);
                const uint32_t b1 = pos + 1 < len ? __ldg(buf + pos + 1) : 0u;
                sv = lds_u8(first_addr + b) && (pos + 1 < len || !open_end ? second_byte_ok(b, b1) : true);
            }
            push(sv, pos);
        }
        for (int64_t base = tail; base < W.start_hi; base += 32) {
            const int64_t pos = base + lane;
            bool sv = false;
            if (pos < W.start_hi) {
                const uint32_t b = __ldg(buf + pos);
                const uint32_t b1 = pos + 1 < len ? __ldg(buf + pos + 1) : 0u;
                sv = lds_u8(first_addr + b) && (pos + 1 < len || !open_end ? second_byte_ok(b, b1) : true);
            }
            push(sv, pos);
        }
    }
    for (int64_t u0 = gwarp * 32; u0 < nvec; u0 += nwarps * 32) {
        unsigned long long cur = 0;
        if (lane == 0) cur = *reinterpret_cast<volatile unsigned long long*>(best);
        cur = __shfl_sync(FULL, cur, 0);
        if (cur != NO_START && (unsigned long long)(W.origin + head + (u0 << 4)) + 2 > cur) break;   // behind the winner
        const int64_t u = u0 + lane;
        const bool valid = u < nvec;
        const int64_t pos0 = head + (u << 4);
        uint4 v = make_uint4(0, 0, 0, 0);
        if (valid) v = ldg_nc_v4(buf + pos0);
        const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
        uint32_t hits = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) {
#pragma unroll
            for (int r = 0; r < 4; r++) hits |= lds_u8(first_addr + ((wv[q] >> (8 * r)) & 0xFF)) << (q * 4 + r);
        }
        if (!valid) hits = 0;
        // byte that follows this unit: the next lane's first byte, or a load for the last lane / last unit
        uint32_t follow = __shfl_down_sync(FULL, v.x & 0xFF, 1);
        const bool has_follow = pos0 + 16 < len;
        if (valid && (lane == 31 || u + 1 >= nvec)) follow = has_follow ? __ldg(buf + pos0 + 16) : 0u;
        while (__any_sync(FULL, hits != 0)) {
            bool sv = false;
            int64_t pos = 0;
            if (hits) {
                const int k = __ffs(hits) - 1;
                hits &= hits - 1;
                pos = pos0 + k;
                const uint32_t b = (wv[k >> 2] >> (8 * (k & 3))) & 0xFF;
                const uint32_t b1 = k < 15 ? (wv[(k + 1) >> 2] >> (8 * ((k + 1) & 3))) & 0xFF : follow;
                const bool know_b1 = k < 15 || has_follow || !open_end;   // at an open window end the next byte is unknown
                sv = know_b1 ? second_byte_ok(b, b1) : true;
            }
            push(sv, pos);
        }
    }
    if (qn > 0) run_batch(qn);
}

// K4 with the SWAR first-byte filter of K2c, for patterns whose set F of possible first bytes is small (C4: the
// bytes that `^` can consume).  Same result as k_buffer_scan -- the smallest start whose anchored attempt wins -- but
// the sweep costs a few integer instructions per 4 bytes instead of one shared-memory lookup per byte:
//   sweep   warps take groups of 4 rows x 32 lanes x 32 bytes (4 KB in flight per warp), front to back, and stop
//           behind the best start found so far; 32-byte units that may hold a candidate are queued per warp;
//   units   32 at a time, one per lane: per-byte candidate mask, candidates confirmed in rounds by the first two
//           table steps (an open window end leaves the second undecided); survivors are queued;
//   starts  32 at a time: boundary check + anchored attempt from global memory (try_start), 64-bit atomicMin.
// shared memory: classmap 256 | table | 8 warps x (unit queue 64 x int64 | start queue 64 x int64)
__host__ __device__ __forceinline__ int scan_sparse_smem_bytes(int table_smem_bytes) {
    return ((256 + table_smem_bytes + 15) & ~15) + 8 * 2 * 64 * 8;
}

//
// PREFIX: the pattern has an extracted prefix literal and the reference takes its candidate starts from the
// occurrences of that literal in the text (api_internal_m.F90:76-104, utility_m.f90:58-117) instead of from every
// character boundary.  The host takes this form only for a prefix without border (its occurrences cannot overlap, so
// "non-overlapping occurrences, left to right" is simply "all occurrences") and an empty suffix.  The sweep looks for
// the literal's first byte, the unit phase compares the whole literal, and best[2] counts the occurrences seen: when
// the literal occurs nowhere the reference falls back to all boundaries -- the caller then runs the plain scan, which
// is gated on best[2] == 0.  The start on the leading NUL is tried iff the literal sits at the very front of the text.
template <int KIND, int NR, bool HIGH, bool PREFIX>
__global__ void __launch_bounds__(256) k_buffer_scan_sparse(KParams p, SparseParams sp, const uint8_t* __restrict__ buf,
                                                            ScanWindow W, unsigned long long* __restrict__ best,
                                                            int table_smem_bytes, const unsigned long long* __restrict__ gate,
                                                            const unsigned long long* __restrict__ run_if, ScanBudget B) {
    if (gate != nullptr && *gate != 0) return;      // (plain scan of a prefix pattern) the prefix occurs in the text
    if (run_if != nullptr && *run_if == 0) return;  // fallback behind the state-map scan: only if that scan declined
    uint32_t acc = 0;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_cmap = smem;
    uint8_t* s_table = smem + 256;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int64_t* s_units = reinterpret_cast<int64_t*>(smem + ((256 + table_smem_bytes + 15) & ~15)) + warp * 128;
    int64_t* s_starts = s_units + 64;
    Table<KIND> T = stage_table<KIND>(p, s_table, s_cmap);
    __syncthreads();
    const uint32_t q0 = (uint32_t)p.q0;
    const int64_t len = W.len;
    const bool open_end = !W.last;
    unsigned long long* overflow = best + 1;
    const uint32_t FULL = 0xffffffffu;
    const uint8_t* pre = p.lits + p.all_len;                // PREFIX: the literal
    const int plen = p.pre_len;
    auto prefix_at = [&](int64_t pos) -> int {              // 1: the literal is at pos; 0: it is not; -1: the window ends first
        if (pos + plen > len) return open_end ? -1 : 0;
        for (int k = 0; k < plen; k++)
            if (__ldg(buf + pos + k) != __ldg(pre + k)) return 0;
        return 1;
    };
    if (blockIdx.x == 0 && threadIdx.x == 0 && W.first) {   // start 1 = the leading NUL sentinel
        const Anchored A{p.flags, p.start_nul, p.q0};
        if (!PREFIX || (W.start_lo == 0 && prefix_at(0) == 1))
            if (attempt_at(A, T, FetchGlobal{buf}, len, 1) >= 0) atomicMin(best, 1ull);
    }
    const uintptr_t gbuf = reinterpret_cast<uintptr_t>(buf);
    const uintptr_t ubase = (gbuf + (uintptr_t)W.start_lo) & ~(uintptr_t)31;      // 32-byte units aligned to the buffer ADDRESS
    const int64_t nunits = W.start_hi > W.start_lo ? (int64_t)((gbuf + (uintptr_t)W.start_hi - ubase + 31) >> 5) : 0;
    const int64_t pos_base = (int64_t)ubase - (int64_t)gbuf;                      // window position of unit 0's first byte (may be < start_lo)
    int uqn = 0, sqn = 0;

    auto run_starts = [&](int count) {
        __syncwarp();
        if (B.limit != 0) {                                  // the budget is spent: no more attempts from this scan
            unsigned long long ab = 0;
            if (lane == 0) ab = *reinterpret_cast<volatile unsigned long long*>(B.abort);
            if (__shfl_sync(FULL, ab, 0) != 0) return;
        }
        if (lane < count) {
            const int64_t pos = s_starts[lane];
            if (try_start(p, T, buf, len, pos, __ldg(buf + pos), open_end, overflow, B, acc))
                atomicMin(best, (unsigned long long)(W.origin + pos) + 2);
        }
        __syncwarp();
    };
    auto run_units = [&](int count) {
        __syncwarp();
        uint32_t cand = 0;
        int64_t P = 0;
        if (lane < count) {
            const int64_t u = s_units[lane];
            const uintptr_t ua = ubase + ((uintptr_t)u << 5);
            const uint4 v0 = __ldg(reinterpret_cast<const uint4*>(ua)), v1 = __ldg(reinterpret_cast<const uint4*>(ua + 16));
            cand = pack_byte_flags(first_mask<NR, HIGH>(sp, v0.x)) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v0.y)) << 4) |
                   (pack_byte_flags(first_mask<NR, HIGH>(sp, v0.z)) << 8) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v0.w)) << 12) |
                   (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.x)) << 16) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.y)) << 20) |
                   (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.z)) << 24) | (pack_byte_flags(first_mask<NR, HIGH>(sp, v1.w)) << 28);
            P = pos_base + (u << 5);
            if (P < W.start_lo) cand &= 0xFFFFFFFFu << (int)(W.start_lo - P);
            if (P + 32 > W.start_hi) cand &= (P >= W.start_hi) ? 0u : (0xFFFFFFFFu >> (int)(P + 32 - W.start_hi));
        }
        while (__any_sync(FULL, cand != 0)) {
            bool sv = false;
            int64_t pos = 0;
            if (cand && PREFIX) {
                pos = P + __ffs(cand) - 1;
                cand &= cand - 1;
                const int occ = prefix_at(pos);
                if (occ < 0) atomicAdd(overflow, 1ull);              // cannot be decided in this window
                if (occ > 0) { best[2] = 1; sv = true; }
            } else if (cand) {
                pos = P + __ffs(cand) - 1;
                cand &= cand - 1;
                // up to four plain steps: a start survives unless they prove it dead (undecided -- an accept, a multi-byte
                // sequence, the end of the window -- keeps it).  Four rather than two so that what reaches the attempt
                // phase is uniformly long-lived (C4: `CR LF I...` dies here, only ERROR lines go on).
                uint32_t st = q0;
                int64_t q = pos;
                sv = true;
                for (int k = 0; k < 4 && q < len; k++, q++) {
                    const uint32_t nw = T.next(st, __ldg(buf + q));
                    if (nw & (W_ACC | W_INTER)) break;
                    if (nw == 0) { sv = false; break; }
                    st = nw;
                }
                if (sv && q >= len && !open_end && (st & (W_ACC | W_INTER)) == 0 && st != q0)   // only the trailing NUL is left
                    sv = (T.next(st, 0u) & (W_STATE | W_ACC)) != 0;
            }
            const uint32_t m = __ballot_sync(FULL, sv);
            if (m) {
                if (sv) s_starts[sqn + __popc(m & ((1u << lane) - 1))] = pos;
                sqn += __popc(m);
                if (sqn >= 32) {
                    run_starts(32);
                    if (lane < sqn - 32) { const int64_t x = s_starts[32 + lane]; s_starts[lane] = x; }
                    sqn -= 32;
                    __syncwarp();
                }
            }
        }
    };

    const int64_t gwarp = (int64_t)blockIdx.x * 8 + warp, nwarps = (int64_t)gridDim.x * 8;
    int sweep_iter = 0;
    for (int64_t g0 = gwarp * 128; g0 < nunits; g0 += nwarps * 128) {
        unsigned long long cur = 0;
        if (lane == 0) cur = *reinterpret_cast<volatile unsigned long long*>(best);
        cur = __shfl_sync(FULL, cur, 0);
        if (cur != NO_START && (unsigned long long)(W.origin + pos_base + (g0 << 5)) + 2 > cur) break;   // behind the winner
        if (B.limit != 0 && (sweep_iter++ & 7) == 0) {       // budget spent somewhere: this scan is over (looked at every 8th group)
            unsigned long long ab = 0;
            if (lane == 0) ab = *reinterpret_cast<volatile unsigned long long*>(B.abort);
            if (__shfl_sync(FULL, ab, 0) != 0) return;
        }
        uint4 va[4], vb[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int64_t u = g0 + k * 32 + lane;
            va[k] = make_uint4(0, 0, 0, 0); vb[k] = va[k];
            if (u < nunits) {
                va[k] = ldg_v4(reinterpret_cast<const void*>(ubase + ((uintptr_t)u << 5)));
                vb[k] = ldg_v4(reinterpret_cast<const void*>(ubase + ((uintptr_t)u << 5) + 16));
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int64_t u = g0 + k * 32 + lane;
            uint32_t seen = 0;
            const bool hit = u < nunits && unit_any<NR, HIGH, false>(sp, va[k], vb[k], seen) != 0;
            const uint32_t m = __ballot_sync(FULL, hit);
            if (hit) s_units[uqn + __popc(m & ((1u << lane) - 1))] = u;
            uqn += __popc(m);
            if (uqn >= 32) {
                run_units(32);
                if (lane < uqn - 32) { const int64_t x = s_units[32 + lane]; s_units[lane] = x; }
                uqn -= 32;
                __syncwarp();
            }
        }
    }
    if (uqn > 0) run_units(uqn);
    if (sqn > 0) run_starts(sqn);
}

// ---------------------------------------------------------------------------------------------
// K5: one long buffer in LINEAR time -- the chunked state-map scan.
// K4 above runs the reference's own loop (one anchored attempt per candidate start) in parallel; its work is the sum of
// the attempt lengths, which is unbounded on text whose attempts run long ([a].*b over a megabyte of `a`).  K5 walks the
// text ONCE with the forward "ordered groups" automaton of the span path (fx_automata.cpp build_span_forward): the last
// position at which that automaton holds the exit is the end of Forgex's leftmost-longest match.  A DFA walk is a
// prefix computation over state maps, so it parallelises:
//   sub-chunks   a lane walks SUB bytes from a small CANDIDATE set of states that provably holds the state the true walk
//                arrives in: the image of ALL reachable states under the byte in front of the sub-chunk (host table
//                `img`, at most 4 live states for most bytes; one more byte back when that byte's image is wide).
//                Candidates that reach the same state merge (checked every 16 bytes); after a few bytes one trajectory
//                is left.  Result: a map candidate -> (end state, last accept).  An accept while candidates still
//                differ, or a byte context whose image is wide, makes the map "unknown";
//   chain        the 32 lanes of a warp chain their maps in text order (maps are broadcast through shared memory);
//                the warp carries up to 32 chain states side by side -- the region's own candidates -- and a chain
//                state that meets an unknown map simply walks that sub-chunk itself (all lanes in parallel);
//   regions      a warp owns a contiguous region (many segments of 32 sub-chunks).  Its candidates come from a full
//                enumeration: every reachable state is walked over the 64 bytes in front of the region and the
//                distinct survivors (<= 32, else the scan declines) are the keys of the region's map;
//   compose      one warp applies the region maps in order, starting from the automaton's start state
//                (k_statemap_compose).  No text is read twice, nothing is quadratic.
// The start of the match comes from one backward walk of the reverse automaton (k_buffer_finish_span).
// Model + proof by fuzz of the candidate argument: tests/table_model.py StateMapScan.
// ---------------------------------------------------------------------------------------------
static constexpr int SM_SUB = 512;               // bytes per lane and segment
static constexpr int SM_M = 4;                   // candidates per sub-chunk
static constexpr int SM_LOOKBACK = 64;           // bytes in front of a region over which every reachable state is walked
static constexpr int SM_WARPS = 16;
static constexpr int SM_SCAN = 256;              // how far behind its nominal start a sub-chunk looks for a synchronising byte (<= SM_SUB)
struct StateMapParams {
    const uint16_t* reach;      // reachable live states of the forward automaton
    const uint16_t* img;        // 256 x (1 + SM_M): count (0xFFFF = more than SM_M) then the live image states of the byte
    const uint8_t* sync;        // 256: 1 = a SYNCHRONISING byte: whatever state reads it and then any one more byte ends up
                                //      in at most one live state, so a walk that starts right behind it is a single
                                //      trajectory within a byte or two (C4: every line end)
    int nreach;
    int64_t region_bytes;       // multiple of 32 * SM_SUB
    int64_t nregions;
    uint16_t* rc;               // nregions x 32: region candidates (0xFFFF = unused lane; all 0xFFFF = the region declined)
    uint16_t* re;               // nregions x 32: end state per candidate
    long long* rl;              // nregions x 32: last accept (text position, -1 none) per candidate
    long long* result;          // [0] = last accept of the whole text (-1 none), [1] = status (0 ok, 1 declined);
                                // window form: the slab map (FX_STATEMAP_MAP_WORDS words, see k_statemap_compose)
    int64_t back;               // bytes of the text in front of buf[0] that the first region may read (<= SM_LOOKBACK);
                                // 0: buf begins the text, and the walk starts in the automaton's start state
    int64_t pos0;               // text position of buf[0]: added to every last accept, so slab maps speak whole-text positions
};
static constexpr long long SM_NO_ACCEPT = -(1ll << 62);     // "no accept yet": in a slab an accept may lie up to 2 bytes
                                                            // in front of buf (a replay across the cut), so -1 is a position
static constexpr long long SM_MAP_UNKNOWN = -2;             // slab map: this key met a region that does not know it

// one forward step on 64-bit positions
#define FX_SM_STEP(T, st, last, b, jj)                                            \
    {                                                                             \
        const uint32_t nw_ = (T).next((st), (b));                                 \
        if (nw_ & 0xB000u) {                                                      \
            if (nw_ & W_RA) (last) = (jj) + 1 - (long long)((nw_ >> 12) & 3u);    \
            if (nw_ & W_ACC) (last) = (jj) + 1;                                   \
        }                                                                         \
        (st) = nw_ & W_SSTATE;                                                    \
    }

// a lane's map for one sub-chunk, as it sits in shared memory
struct SubMap {
    long long b, e;             // the sub-chunk's bytes [b, e)
    uint16_t cand[SM_M];
    uint16_t end[SM_M];
    int32_t last;               // position relative to the sub-chunk's first byte (may be -2..SM_SUB), INT32_MIN = none
    uint16_t owner_mask;        // candidates that follow the trajectory the accepts belong to
    uint8_t ncand;              // 0xFF = unknown: whoever arrives walks the sub-chunk
    uint8_t pad;
};

// WINDOW: buf is a slab that may not begin the text (mp.back, mp.pos0); the whole-text form compiles without them
template <int FK, bool WINDOW>
__global__ void __launch_bounds__(SM_WARPS * 32, 2) k_statemap_regions(SpanParams sp, StateMapParams mp,
                                                                      const uint8_t* __restrict__ buf, int64_t len, int fwd_bytes,
                                                                      const unsigned long long* __restrict__ run_if) {
    if (run_if != nullptr && *run_if == 0) return;            // the budgeted candidate scan has answered
    const int64_t back = WINDOW ? mp.back : 0;
    constexpr long long NO_ACC = WINDOW ? SM_NO_ACCEPT : -1;   // "no accept yet"
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t FULL = 0xffffffffu;
    SpanFwd<FK> T;
    T.s_cmap = smem_u32(smem); T.s_table = smem_u32(smem + 256); T.g_table = sp.table; T.g_cmap = sp.classmap; T.shift = sp.row_shift;
    if (FK == 0) {
        uint16_t* dst = reinterpret_cast<uint16_t*>(smem + 256);
        for (int i = threadIdx.x; i < sp.nstates * 128; i += blockDim.x) {
            const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(sp.direct) + i);
            *reinterpret_cast<uint32_t*>(dst + (i >> 7) * SPAN_ROW + ((i & 127) << 1)) = v;
        }
    } else if (FK == 1) {
        uint32_t* dst = reinterpret_cast<uint32_t*>(smem + 256);
        const int words32 = ((sp.nstates << sp.row_shift) + 1) >> 1;
        for (int i = threadIdx.x; i < words32; i += blockDim.x) dst[i] = __ldg(reinterpret_cast<const uint32_t*>(sp.table) + i);
        for (int i = threadIdx.x; i < 64; i += blockDim.x)
            reinterpret_cast<uint32_t*>(smem)[i] = __ldg(reinterpret_cast<const uint32_t*>(sp.classmap) + i);
    }
    const int head = (256 + fwd_bytes + 15) & ~15;
    uint16_t* s_img = reinterpret_cast<uint16_t*>(smem + head);                          // 256 x 5 x u16
    for (int i = threadIdx.x; i < 256 * (1 + SM_M); i += blockDim.x) s_img[i] = __ldg(mp.img + i);
    uint8_t* s_sync = smem + head + 256 * (1 + SM_M) * 2;
    for (int i = threadIdx.x; i < 64; i += blockDim.x) reinterpret_cast<uint32_t*>(s_sync)[i] = __ldg(reinterpret_cast<const uint32_t*>(mp.sync) + i);
    SubMap* s_maps = reinterpret_cast<SubMap*>(smem + head + 256 * (1 + SM_M) * 2 + 256) + warp * 32;
    uint16_t* s_rc = reinterpret_cast<uint16_t*>(smem + head + 256 * (1 + SM_M) * 2 + 256 + SM_WARPS * 32 * sizeof(SubMap)) + warp * 32;
    __syncthreads();
    const uintptr_t gbuf = reinterpret_cast<uintptr_t>(buf);
    const int64_t shift = (int64_t)(gbuf & 15);          // nominal start of sub-chunk k: text index k * SUB - shift (a 16-byte aligned ADDRESS)
    // Where sub-chunk k really starts: right behind the first synchronising byte at or after its nominal start's
    // predecessor (within SM_SCAN bytes), else at the nominal start.  Every lane computes the same function of the text,
    // so neighbours agree on their common boundary without talking.
    auto bnd = [&](int64_t k) -> int64_t {
        if (k <= 0) return 0;
        const int64_t nom = k * SM_SUB - shift;
        if (nom >= len) return len;
        int64_t lim = nom - 1 + SM_SCAN;
        if (lim > len) lim = len;
        // (same answer as the byte loop `for q = nom - 1 .. lim - 1: if sync[text[q]] return q + 1`, 16 bytes per load:
        //  byte by byte this search was a chain of dependent L1 hits, a fifth of a lane's time on C4)
        int64_t q = nom - 1;
        if (s_sync[__ldg(buf + q)]) return q + 1;
        q = nom;                                              // a 16-byte aligned address from here on
        for (; q + 16 <= lim; q += 16) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(gbuf + (uintptr_t)q));
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
            uint32_t m = 0;
#pragma unroll
            for (int i = 0; i < 16; i++) m |= (uint32_t)s_sync[(w4[i >> 2] >> (8 * (i & 3))) & 0xFFu] << i;
            if (m) return q + __ffs(m);
        }
        for (; q < lim; q++) if (s_sync[__ldg(buf + q)]) return q + 1;
        return nom;
    };
    // bytes [lo, hi) of one 16-byte block, from registers
    auto walk_block = [&](const uint4& v, int lo, int hi, uint32_t& cur, long long& l2, int64_t base) {
        const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 16; i++) {
            if (i >= lo && i < hi) { const uint32_t byte = (w4[i >> 2] >> (8 * (i & 3))) & 0xFFu; FX_SM_STEP(T, cur, l2, byte, base + i); }
        }
    };
    const int64_t spr = mp.region_bytes / SM_SUB;         // sub-chunks per region
    const int64_t gwarp = (int64_t)blockIdx.x * SM_WARPS + warp, nwarps = (int64_t)gridDim.x * SM_WARPS;
    for (int64_t reg = gwarp; reg < mp.nregions; reg += nwarps) {
        const int64_t kr0 = reg * spr, kr1 = (reg + 1) * spr;
        const int64_t r0 = bnd(kr0);
        int64_t r1 = bnd(kr1);
        if (r1 > len) r1 = len;
        // ---- region candidates: every reachable state walked over the look-back window, distinct survivors ----
        int cnt = 0;
        bool wide = false;
        __syncwarp();
        if (r0 == 0 && back == 0) {
            if (lane == 0) s_rc[0] = (uint16_t)sp.start;
            cnt = 1;
        } else {
            const int64_t w0 = r0 - SM_LOOKBACK > -back ? r0 - SM_LOOKBACK : -back;
            for (int k = 0; k < mp.nreach && !wide; k += 32) {
                uint32_t st = k + lane < mp.nreach ? (uint32_t)__ldg(mp.reach + k + lane) : 0u;
                for (int64_t j = w0; j < r0; j++) st = T.next(st, (uint32_t)__ldg(buf + j)) & W_SSTATE;
                const uint32_t peers = __match_any_sync(FULL, st);
                bool isnew = st != 0 && (__ffs(peers) - 1) == lane;
                for (int i = 0; i < cnt; i++) if (s_rc[i] == st) isnew = false;
                const uint32_t m = __ballot_sync(FULL, isnew);
                if (cnt + __popc(m) > 32) { wide = true; break; }
                if (isnew) s_rc[cnt + __popc(m & ((1u << lane) - 1))] = (uint16_t)st;
                cnt += __popc(m);
                __syncwarp();
            }
        }
        __syncwarp();
        if (wide) {                                          // the scan declines: too many states can arrive here
            mp.rc[reg * 32 + lane] = 0xFFFFu; mp.re[reg * 32 + lane] = 0; mp.rl[reg * 32 + lane] = -1;
            continue;
        }
        const uint32_t mycand = lane < cnt ? (uint32_t)s_rc[lane] : 0u;
        uint32_t c = mycand;                                 // this lane's chain state
        long long L = NO_ACC;                                // its last accept
        // ---- segments of 32 sub-chunks ----
        for (int64_t k0 = kr0; k0 < kr1; k0 += 32) {
            const int64_t kb = k0 + lane;
            int64_t b = kb < kr1 ? bnd(kb) : r1;
            if (b > r1) b = r1;
            int64_t e = __shfl_down_sync(FULL, b, 1);
            if (lane == 31) { e = kb + 1 < kr1 ? bnd(kb + 1) : r1; if (e > r1) e = r1; }
            if (__ballot_sync(FULL, b < e) == 0) break;              // behind the end of the text
            SubMap mine;
            mine.b = b; mine.e = e;
            mine.ncand = 0; mine.last = INT32_MIN; mine.owner_mask = 0; mine.pad = 0;
#pragma unroll
            for (int k = 0; k < SM_M; k++) { mine.cand[k] = 0; mine.end[k] = 0; }
            if (b < e) {
                // ---- candidates ----
                uint32_t st[SM_M] = {0, 0, 0, 0};
                int nc = 0;
                bool unknown = false;
                if (b == 0 && back == 0) { st[0] = (uint32_t)sp.start; nc = 1; }
                else {
                    const uint32_t c1 = __ldg(buf + b - 1);
                    const uint32_t n1 = s_img[c1 * (1 + SM_M)];
                    if (n1 <= SM_M) {
                        nc = (int)n1;
#pragma unroll
                        for (int k = 0; k < SM_M; k++) if (k < nc) st[k] = s_img[c1 * (1 + SM_M) + 1 + k];
                    } else if (b + back >= 2) {
                        const uint32_t c2 = __ldg(buf + b - 2);
                        const uint32_t n2 = s_img[c2 * (1 + SM_M)];
                        if (n2 <= SM_M) {
#pragma unroll
                            for (int k = 0; k < SM_M; k++) {
                                if (k < (int)n2) {
                                    const uint32_t v = T.next((uint32_t)s_img[c2 * (1 + SM_M) + 1 + k], c1) & W_SSTATE;
                                    bool dup = v == 0;
#pragma unroll
                                    for (int q = 0; q < SM_M; q++) if (q < nc && st[q] == v) dup = true;
                                    if (!dup) {
#pragma unroll
                                        for (int q = 0; q < SM_M; q++) if (q == nc) st[q] = v;
                                        nc++;
                                    }
                                }
                            }
                        } else unknown = true;
                    } else unknown = true;
                }
                if (unknown) mine.ncand = 0xFF;
                else {
                    mine.ncand = (uint8_t)nc;
#pragma unroll
                    for (int k = 0; k < SM_M; k++) mine.cand[k] = (uint16_t)st[k];
                    // ---- walk: all candidates until they have merged, 16 bytes between merge checks ----
                    uint32_t active = 0, root = 0x3210u;     // bit k: candidate k is walked; nibble k of root: whom k follows
#pragma unroll
                    for (int k = 0; k < SM_M; k++) if (k < nc && st[k] != 0) active |= 1u << k;
                    long long last = NO_ACC;
                    int owner = -1;
                    bool complex = false;
                    int64_t j = b;
                    while (j < e && (active & (active - 1)) != 0 && !complex) {     // phase 1: several trajectories, 16 bytes between merge checks
                        int nb = (int)(e - j < 16 ? e - j : 16);
                        const uintptr_t ga = gbuf + (uintptr_t)j;
                        uint32_t w[4];
                        if ((ga & 15) == 0 && nb == 16) {
                            const uint4 v = __ldg(reinterpret_cast<const uint4*>(ga));
                            w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
                        } else {                             // the first block of the text / the last of the region: bytes
                            const int room = (int)(16 - (ga & 15));
                            if (nb > room) nb = room;
                            w[0] = w[1] = w[2] = w[3] = 0;
                            for (int i = 0; i < nb; i++) w[i >> 2] |= (uint32_t)__ldg(buf + j + i) << (8 * (i & 3));
                        }
#pragma unroll
                        for (int i = 0; i < 16; i++) {
                            if (i < nb) {
                                const uint32_t byte = (w[i >> 2] >> (8 * (i & 3))) & 0xFFu;
#pragma unroll
                                for (int k = 0; k < SM_M; k++) {
                                    if (active & (1u << k)) {
                                        const uint32_t nw = T.next(st[k], byte);
                                        if (nw & 0xB000u) {
                                            if (active & (active - 1)) complex = true;       // an accept while trajectories still differ
                                            owner = k;
                                            if (nw & W_RA) last = j + i + 1 - (long long)((nw >> 12) & 3u);
                                            if (nw & W_ACC) last = j + i + 1;
                                        }
                                        st[k] = nw & W_SSTATE;
                                        if (st[k] == 0) active &= ~(1u << k);
                                    }
                                }
                            }
                        }
                        j += nb;
                        if (active & (active - 1)) {          // merge check
#pragma unroll
                            for (int k = 1; k < SM_M; k++) {
#pragma unroll
                                for (int m = 0; m < k; m++) {
                                    if ((active & (1u << k)) && (active & (1u << m)) && st[k] == st[m]) {
                                        active &= ~(1u << k);
#pragma unroll
                                        for (int q = 0; q < SM_M; q++)
                                            if (((root >> (4 * q)) & 15u) == (uint32_t)k) root = (root & ~(15u << (4 * q))) | ((uint32_t)m << (4 * q));
                                    }
                                }
                            }
                        }
                    }
                    if (!complex && active != 0 && j < e) {
                        // phase 2: ONE trajectory is left (the usual state a few bytes into the sub-chunk).  Four steps run
                        // without looking at the flag bits; the OR of the four words is tested once and only a word that
                        // held an event is walked again with the books.
                        const int k1 = __ffs(active) - 1;
                        uint32_t cur = k1 == 0 ? st[0] : k1 == 1 ? st[1] : k1 == 2 ? st[2] : st[3];
                        long long l2 = NO_ACC;
                        // (whole aligned 16-byte blocks are loaded even where only part of one belongs to the sub-chunk:
                        //  a block that holds one byte of the text lies inside the text's allocation)
                        if ((gbuf + (uintptr_t)j) & 15) {                        // head: up to the next 16-byte boundary
                            const int lo = (int)((gbuf + (uintptr_t)j) & 15);
                            const int hi = e - j < 16 - lo ? lo + (int)(e - j) : 16;
                            const uint4 v = __ldg(reinterpret_cast<const uint4*>((gbuf + (uintptr_t)j) & ~(uintptr_t)15));
                            walk_block(v, lo, hi, cur, l2, j - lo);
                            j += hi - lo;
                        }
                        if (cur != 0 && j + 16 <= e) {                           // whole blocks, the next one in flight
                            uint4 v = __ldg(reinterpret_cast<const uint4*>(gbuf + (uintptr_t)j));
                            for (;;) {
                                const bool more = j + 32 <= e;
                                uint4 vn = make_uint4(0, 0, 0, 0);
                                if (more) vn = __ldg(reinterpret_cast<const uint4*>(gbuf + (uintptr_t)j + 16));
                                const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                                for (int q = 0; q < 4; q++) {
                                    const uint32_t n1 = T.next(cur, w4[q] & 0xFFu);
                                    const uint32_t n2 = T.next(n1 & W_SSTATE, (w4[q] >> 8) & 0xFFu);
                                    const uint32_t n3 = T.next(n2 & W_SSTATE, (w4[q] >> 16) & 0xFFu);
                                    const uint32_t n4 = T.next(n3 & W_SSTATE, w4[q] >> 24);
                                    if ((n1 | n2 | n3 | n4) & 0xB000u) {
                                        const long long jj = j + 4 * q;
                                        FX_SPAN_BOOKS4(n1, n2, n3, n4, l2, jj);
                                    }
                                    cur = n4 & W_SSTATE;
                                }
                                j += 16;
                                if (!more || cur == 0) break;
                                v = vn;
                            }
                        }
                        if (cur != 0 && j < e) {                                 // tail: part of one more block (j is aligned here)
                            const uint4 v = __ldg(reinterpret_cast<const uint4*>(gbuf + (uintptr_t)j));
                            walk_block(v, 0, (int)(e - j), cur, l2, j);
                            j = e;
                        }
                        if (WINDOW ? l2 != NO_ACC : l2 >= 0) { last = l2; owner = k1; }
#pragma unroll
                        for (int k = 0; k < SM_M; k++) if (k == k1) st[k] = cur;
                        if (cur == 0) active = 0;
                    }
                    if (complex) mine.ncand = 0xFF;
                    else {
                        uint32_t om = 0;
#pragma unroll
                        for (int k = 0; k < SM_M; k++) {
                            const uint32_t r = (root >> (4 * k)) & 15u;
                            uint32_t es = 0;
#pragma unroll
                            for (int q = 0; q < SM_M; q++) if (q == (int)r) es = st[q];
                            mine.end[k] = (uint16_t)es;
                            if ((int)r == owner) om |= 1u << k;
                        }
                        mine.owner_mask = (uint16_t)om;
                        mine.last = (WINDOW ? last != NO_ACC : last >= 0) ? (int32_t)(last - b) : INT32_MIN;
                    }
                }
            }
            s_maps[lane] = mine;
            __syncwarp();
            // ---- chain the 32 maps in text order; every lane carries its own chain state ----
            for (int t = 0; t < 32; t++) {
                const SubMap m = s_maps[t];
                const int64_t tb = m.b, te = m.e;
                if (tb >= te) continue;
                bool need = false;
                if (c != 0) {
                    int hit = -1;
                    if (m.ncand != 0xFF) {
#pragma unroll
                        for (int k = 0; k < SM_M; k++) if (k < m.ncand && m.cand[k] == c) hit = k;
                    }
                    if (hit >= 0) {
                        c = m.end[hit];
                        if (m.last != INT32_MIN && ((m.owner_mask >> hit) & 1u)) L = tb + m.last;
                    } else need = true;
                }
                if (__any_sync(FULL, need)) {                 // unknown map (or, never, a missing key): walk the sub-chunk
                    if (need) for (int64_t j = tb; j < te && c != 0; j++) { const uint32_t byte = __ldg(buf + j); FX_SM_STEP(T, c, L, byte, j); }
                }
            }
            __syncwarp();
        }
        mp.rc[reg * 32 + lane] = lane < cnt ? (uint16_t)mycand : (uint16_t)0xFFFFu;
        mp.re[reg * 32 + lane] = (uint16_t)c;
        mp.rl[reg * 32 + lane] = WINDOW ? (L == NO_ACC ? -1 : L + mp.pos0) : L;
    }
}

// Apply the region maps in order.  The chain is a composition of (partial) maps, so it is done in two levels: each of
// the 32 warps composes a contiguous RANGE of regions -- lane k carries the k-th candidate of the range's first region
// through the range (a lookup among a region's 32 keys is 32 shuffles; eight regions' maps are fetched at a time) --
// and warp 0 then chains the 32 range maps from the automaton's start state.  (One warp walking the ~19 000 regions of
// a multi-GiB text one after the other took 13 ms, 4.2 ms with batched loads; this form takes a few hundred us.)
// WINDOW: buf is a slab of a text split across GPUs.  The true state at the slab's start is unknown here, so warp 0
// chains the 32 range maps for EVERY key of region 0 (one per lane) and writes the slab map to mp.result:
//   [0] status (0 ok, 1 declined, 2 empty slab), [1] key count, [2..33] keys, [34..65] end states,
//   [66..97] last accepts in text positions (-1 none, SM_MAP_UNKNOWN: the key met a region that does not know it).
// No end-of-text step: fx_statemap_combine applies it after the last slab.
template <bool WINDOW>
__global__ void __launch_bounds__(1024) k_statemap_compose(SpanParams sp, StateMapParams mp, int64_t len,
                                                           const unsigned long long* __restrict__ run_if) {
    if (run_if != nullptr && *run_if == 0) return;
    if (WINDOW && len == 0) {
        if (threadIdx.x < 32) {
            mp.result[2 + threadIdx.x] = 0; mp.result[34 + threadIdx.x] = 0; mp.result[66 + threadIdx.x] = -1;
            if (threadIdx.x == 0) { mp.result[0] = 2; mp.result[1] = 0; }
        }
        return;
    }
    __shared__ uint16_t r_key[32][32], r_end[32][32];
    __shared__ long long r_l[32][32];
    __shared__ uint8_t r_bad[32][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t FULL = 0xffffffffu;
    const int64_t n = mp.nregions;
    const int64_t per = (n + 31) / 32;
    const int64_t ra = (int64_t)warp * per < n ? (int64_t)warp * per : n;
    const int64_t rb = ra + per < n ? ra + per : n;
    {
        uint32_t key0 = 0xFFFFu, cs = 0xFFFFu;            // this lane's candidate of the range's first region, its chain state
        long long L = -1;
        bool bad = false;
        if (ra < rb) { key0 = mp.rc[ra * 32 + lane]; cs = key0; }
        constexpr int CB = 8;
        for (int64_t r0 = ra; r0 < rb; r0 += CB) {
            uint32_t key[CB], end[CB];
            long long l[CB];
#pragma unroll
            for (int k = 0; k < CB; k++) {
                const int64_t r = r0 + k < rb ? r0 + k : rb - 1;
                key[k] = mp.rc[r * 32 + lane];
                end[k] = mp.re[r * 32 + lane];
                l[k] = mp.rl[r * 32 + lane];
            }
#pragma unroll
            for (int k = 0; k < CB; k++) {
                if (r0 + k < rb) {                        // (warp-uniform)
                    int hit = -1;
                    for (int q = 0; q < 32; q++) if (__shfl_sync(FULL, key[k], q) == cs) hit = q;
                    const uint32_t e = __shfl_sync(FULL, end[k], hit < 0 ? 0 : hit);
                    const long long ll = __shfl_sync(FULL, l[k], hit < 0 ? 0 : hit);
                    if (cs != 0xFFFFu && cs != 0 && !bad) {
                        if (hit < 0) bad = true;          // the region declined, or does not know this state
                        else { cs = e; if (ll >= 0) L = ll; }
                    }
                }
            }
        }
        r_key[warp][lane] = (uint16_t)key0; r_end[warp][lane] = (uint16_t)cs; r_l[warp][lane] = L; r_bad[warp][lane] = bad ? 1 : 0;
    }
    __syncthreads();
    if (warp != 0) return;
    if (WINDOW) {
        const uint32_t key = r_key[0][lane];
        const bool live = key != 0xFFFFu;
        uint32_t cs = r_end[0][lane];
        long long L = r_l[0][lane];
        bool unknown = r_bad[0][lane] != 0;
        for (int w = 1; w < 32 && live && cs != 0 && !unknown; w++) {
            if ((int64_t)w * per >= n) break;
            int src = -1;
            for (int q = 0; q < 32; q++) if (r_key[w][q] == cs) src = q;
            if (src < 0 || r_bad[w][src]) { unknown = true; break; }
            cs = r_end[w][src];
            if (r_l[w][src] >= 0) L = r_l[w][src];
        }
        const int nkeys = __popc(__ballot_sync(FULL, live));
        if (lane == 0) { mp.result[0] = nkeys == 0 ? 1 : 0; mp.result[1] = nkeys; }   // no key: region 0 declined
        mp.result[2 + lane] = live ? key : 0;
        mp.result[34 + lane] = live && !unknown ? cs : 0;
        mp.result[66 + lane] = !live ? -1 : unknown ? SM_MAP_UNKNOWN : L;
        return;
    }
    uint32_t st = (uint32_t)sp.start;
    long long L = sp.start_acc ? 0 : -1;
    int status = 0;
    for (int w = 0; w < 32 && st != 0 && status == 0; w++) {
        const int64_t wa = (int64_t)w * per;
        if (wa >= n) break;
        const uint32_t m = __ballot_sync(FULL, (uint32_t)r_key[w][lane] == st);
        if (m == 0) { status = 1; break; }                // no answer from this scan
        const int src = __ffs(m) - 1;
        if (r_bad[w][src]) { status = 1; break; }
        st = r_end[w][src];
        const long long ll = r_l[w][src];
        if (ll >= 0) L = ll;
    }
    if (status == 0 && st != 0) {                         // end of the text: pending bytes replay, the trailing NUL is consumed
        const uint32_t e = __ldg(sp.endinfo + st);
        if (e & 3u) L = len + 1 - (long long)(e & 3u);
        if (e & 4u) L = len + 1;
    }
    if (lane == 0) { mp.result[0] = status == 0 ? L : -1; mp.result[1] = status; }
}

// The backward half on 64-bit positions (one thread), as a resumable step loop over (pos, reverse state r, best so far).
// Text byte p is win[p - org].  The loop steps while r lives and pos > 0, and -- unless the window begins the text
// (org == 0) -- only while the next character's decode stays inside the window (pos - 4 >= org): a walk stopped there
// is continued by whoever holds the bytes in front.
__device__ inline void span_back_steps(const SpanParams& sp, const uint8_t* __restrict__ win, long long org, long long& pos,
                                       uint32_t& r, long long& best) {
    SpanRev<false> R;
    R.s_delta = R.s_page = R.s_mixed = 0;
    const uint8_t* buf = win - org;          // (only ever dereferenced at positions >= org)
    while (r != 0 && pos > 0 && (org == 0 || pos - 4 >= org)) {
        uint32_t c = __ldg(buf + pos - 1);
        long long q = pos - 1;
        uint32_t cp = c;
        if (c >= 0x80u) {
            cp = 0xFFFFu;
            if ((c & 0xC0u) == 0x80u && pos >= 2) {
                const uint32_t d1 = __ldg(buf + pos - 2);
                if ((d1 & 0xE0u) == 0xC0u) { cp = ((d1 & 0x1Fu) << 6) | (c & 0x3Fu); q = pos - 2; }
                else if ((d1 & 0xC0u) == 0x80u && pos >= 3) {
                    const uint32_t d2 = __ldg(buf + pos - 3);
                    if ((d2 & 0xF0u) == 0xE0u) { cp = ((d2 & 0x0Fu) << 12) | ((d1 & 0x3Fu) << 6) | (c & 0x3Fu); q = pos - 3; }
                    else if ((d2 & 0xC0u) == 0x80u && pos >= 4) {
                        const uint32_t d3 = __ldg(buf + pos - 4);
                        if ((d3 & 0xF8u) == 0xF0u) {
                            cp = ((d3 & 0x07u) << 18) | ((d2 & 0x3Fu) << 12) | ((d1 & 0x3Fu) << 6) | (c & 0x3Fu);
                            q = pos - 4;
                        }
                    }
                }
            }
        }
        const uint32_t w = R.delta(sp, r, R.cls(sp, cp));
        r = w & 0x7FFFu;
        if (r == 0) break;
        pos = q;
        if (w & 0x8000u) best = pos;
    }
}

// start of the backward walk from the end `last` of the match (the trailing NUL first when it was consumed)
__device__ inline void span_back_begin(const SpanParams& sp, long long len, long long last, long long& pos, uint32_t& r,
                                       long long& best) {
    SpanRev<false> R;
    R.s_delta = R.s_page = R.s_mixed = 0;
    r = (uint32_t)sp.rstart;
    pos = last;
    if (last > len) { r = R.delta(sp, r, (uint32_t)sp.nul_class) & 0x7FFFu; pos = len; }
    best = -2;
}

// end of the backward walk (it stopped, or reached position 0): the leading NUL's step, then `from` (0: none)
__device__ inline long long span_back_end(const SpanParams& sp, long long pos, uint32_t r, long long best) {
    if (r != 0 && pos == 0) {
        SpanRev<false> R;
        R.s_delta = R.s_page = R.s_mixed = 0;
        const uint32_t w = R.delta(sp, r, (uint32_t)sp.nul_class);
        if ((w & 0x7FFFu) != 0 && (w & 0x8000u)) best = -1;
    }
    if (best == -2) return 0;
    return best < 0 ? 1 : best + 1;
}

// the leftmost start of the match that ends at `last`, the whole text in buf
__device__ inline long long span_backward64(const SpanParams& sp, const uint8_t* __restrict__ buf, long long len, long long last) {
    long long pos, best;
    uint32_t r;
    span_back_begin(sp, len, last, pos, r, best);
    span_back_steps(sp, buf, 0, pos, r, best);
    return span_back_end(sp, pos, r, best);
}

// The backward walk of a text split across GPUs (one thread), over the window win[0, wlen) = text[org, org + wlen).
// walk = {pos, best, reverse state, end}: the caller starts it as {0, 0, SM_WALK_NEW, end of the match}; each call
// walks as far as the window allows.  When the walk is over: walk = {from, to, SM_WALK_DONE, end}, exactly
// k_buffer_finish_span's answer for the whole text; otherwise it goes on at the holder of text byte pos - 1.
static constexpr long long SM_WALK_NEW = -1, SM_WALK_DONE = -2;
__global__ void k_statemap_back(SpanParams sp, const uint8_t* __restrict__ win, int64_t org, int64_t wlen, int64_t len,
                                long long* __restrict__ walk) {
    const long long state = walk[2], last = walk[3];
    if (state == SM_WALK_DONE) return;
    long long pos = walk[0], best = walk[1];
    uint32_t r = (uint32_t)state;
    if (state == SM_WALK_NEW) {
        // the blank-text rule (api_internal_m.F90:68-74) and "no match"; a text of one byte lies in every window
        const bool blank = len == 0 || (len == 1 && org == 0 && wlen >= 1 && __ldg(win) == 0x20);
        if (blank || last <= 0) { walk[0] = 0; walk[1] = 0; walk[2] = SM_WALK_DONE; return; }
        span_back_begin(sp, len, last, pos, r, best);
    }
    span_back_steps(sp, win, org, pos, r, best);
    if (r != 0 && pos > 0) { walk[0] = pos; walk[1] = best; walk[2] = r; return; }     // at the window's front edge
    const long long f = span_back_end(sp, pos, r, best);
    walk[0] = f > 0 ? f : 0;
    walk[1] = f > 0 ? (last < len ? last : len) : 0;
    walk[2] = SM_WALK_DONE;
}

// finish of the state-map scan: (from, to) from the end position the compose step found.  `done`: set to 1 when this
// kernel has produced the answer (the fallback scan behind it is then skipped).
__global__ void k_buffer_finish_span(SpanParams sp, const uint8_t* __restrict__ buf, int64_t len, const long long* __restrict__ result,
                                     int64_t* __restrict__ from_to, unsigned long long* __restrict__ done,
                                     unsigned long long* __restrict__ declined, const unsigned long long* __restrict__ run_if,
                                     const uint8_t* __restrict__ lit, int lit_len) {
    if (run_if != nullptr && *run_if == 0) return;
    if (result[1] != 0) { *declined = 1; return; }           // the scan declined: the candidate scan runs again, unbudgeted
    const long long last = result[0];
    long long from = 0, to = 0;
    if (!(len == 0 || (len == 1 && __ldg(buf) == 0x20)) && last > 0) {        // api_internal_m.F90:68-74; to = 0 is "no match"
        const long long f = span_backward64(sp, buf, len, last);
        if (f > 0) { from = f; to = last < len ? last : len; }
    }
    if (lit_len > 0 && from > 0) {
        // a pattern with a prefix literal: Forgex only tries the literal's occurrences.  The winner of "every boundary"
        // is Forgex's winner iff it begins with the literal's own bytes; otherwise (an overlong encoding) decline.
        bool same = from - 1 + lit_len <= len;
        for (int k = 0; k < lit_len && same; k++) same = __ldg(buf + from - 1 + k) == __ldg(lit + k);
        if (!same) { *declined = 1; return; }
    }
    from_to[0] = from; from_to[1] = to;
    *done = 1;
}

// ---------------------------------------------------------------------------------------------
// All matches of a pattern in a text, as a caller of the reference collects them: call regex(), take the match, call
// regex() again on the rest text(to+1:) (README.md:197-222 shows the slicing), until nothing is found.  Every call
// frames ITS text afresh (api_internal_m.F90:55): the rest begins behind a new leading NUL, so `^` matches at every
// restart, and the blank-text rule (api_internal_m.F90:68-74) applies to the rest.  Matches are never empty
// (forgex.F90:332: from > 0 and to > 0), so the loop always advances.
// ---------------------------------------------------------------------------------------------
// one regex() on text[0, len): Forgex's (from, to), (0, 0) = none.  SPAN: the linear-time span path, else the emulation
template <bool SPAN>
__device__ __forceinline__ void regex_once(const KParams& p, const SpanParams& sp, const uint8_t* __restrict__ s, int64_t len,
                                           int64_t& from, int64_t& to) {
    from = 0; to = 0;
    if (SPAN && len < 0x7FFFFFF0ll) {
        if (len == 0 || (len == 1 && __ldg(s) == 0x20)) return;
        SpanFwd<2> T;
        T.s_cmap = T.s_table = 0; T.g_table = sp.table; T.g_cmap = sp.classmap; T.shift = sp.row_shift;
        SpanRev<false> R;
        R.s_delta = R.s_page = R.s_mixed = 0;
        span_linear(sp, T, R, FetchGlobal{s}, (int)len, from, to);
    } else {
        Table<3> G;
        G.g_table = p.ctable; G.g_cmap = p.classmap; G.shift = p.c_row_shift; G.s_table = 0; G.s_cmap = 0;
        eval_regex(p, G, FetchGlobal{s}, len, from, to);
    }
}

// number of matches per string of a ragged batch (one thread per string)
template <bool SPAN>
__global__ void __launch_bounds__(256) k_regex_count(KParams p, SpanParams sp, const uint8_t* __restrict__ buf,
                                                     const int64_t* __restrict__ offsets, int64_t n, int64_t* __restrict__ counts) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o0 = __ldg(offsets + i), o1 = __ldg(offsets + i + 1);
        int64_t pos = 0, cnt = 0;
        for (;;) {
            int64_t f, t;
            regex_once<SPAN>(p, sp, buf + o0 + pos, o1 - o0 - pos, f, t);
            if (f <= 0 || t <= 0) break;
            cnt++;
            pos += t;
        }
        counts[i] = cnt;
    }
}

// The all-matches loop over ONE buffer, its short steps.  state[0] = position of the rest, state[1] = matches so far,
// state[2] = 1 when the loop is over, state[3] = 1 when this kernel gave up on a long search (the host then runs the
// parallel long-buffer search on the rest and comes back).  One thread: from the rest's start the forward automaton is
// walked at most `reach` bytes; a match that completes in that stretch is recorded and the loop goes on, up to
// `max_matches` per launch.  Dense matches are collected here at one launch per thousand; the far ones by K4 / K5.
__global__ void k_buffer_all_local(KParams p, SpanParams sp, const uint8_t* __restrict__ buf, int64_t len, int64_t* __restrict__ state,
                                   int64_t* __restrict__ out_from, int64_t* __restrict__ out_to, int64_t capacity,
                                   int max_matches, int64_t reach) {
    int64_t pos = state[0], cnt = state[1];
    state[3] = 0;
    SpanFwd<2> T;
    T.s_cmap = T.s_table = 0; T.g_table = sp.table; T.g_cmap = sp.classmap; T.shift = sp.row_shift;
    SpanRev<false> R;
    R.s_delta = R.s_page = R.s_mixed = 0;
    for (int it = 0; it < max_matches; it++) {
        const int64_t rem = len - pos;
        const uint8_t* s = buf + pos;
        if (rem == 0 || (rem == 1 && __ldg(s) == 0x20)) { state[2] = 1; break; }      // api_internal_m.F90:68-74: no match
        const int lim = (int)(rem < reach ? rem : reach);
        uint32_t st = (uint32_t)sp.start;
        int last = sp.start_acc ? 0 : -1;
        int j = 0;
        for (; j < lim && st != 0; j++) { const uint32_t b = __ldg(s + j); FX_SPAN_STEP(T, st, last, b, j); }
        if (st != 0 && (int64_t)j < rem) { state[3] = 1; break; }                     // still searching: a job for the parallel scan
        const int ln = rem < 0x7FFFFFF0ll ? (int)rem : 0x7FFFFFF0;                     // (`last` is at most reach + 1 here)
        if (st != 0) last = span_end_of_text(sp, st, ln, last);
        if (last <= 0) { state[2] = 1; break; }                                       // the rest holds no match
        const int f = span_backward(sp, R, FetchGlobal{s}, ln, last);
        const int64_t t = last < rem ? last : rem;
        if (f <= 0) { state[2] = 1; break; }
        if (cnt < capacity) { out_from[cnt] = pos + f; out_to[cnt] = pos + t; }
        cnt++;
        pos += t;
    }
    state[0] = pos; state[1] = cnt;
}
// the far step: the long-buffer search has run on the rest (from_to relative to it): record, advance
__global__ void k_buffer_all_take(const int64_t* __restrict__ from_to, int64_t* __restrict__ state, int64_t* __restrict__ out_from,
                                  int64_t* __restrict__ out_to, int64_t capacity) {
    const int64_t f = from_to[0], t = from_to[1];
    if (f == -2) { state[2] = 1; state[4] = 1; return; }    // the search ran out of its work budget
    if (f <= 0 || t <= 0) { state[2] = 1; return; }
    const int64_t pos = state[0], cnt = state[1];
    if (cnt < capacity) { out_from[cnt] = pos + f; out_to[cnt] = pos + t; }
    state[0] = pos + t; state[1] = cnt + 1;
}

// K4L: a pattern that is ONE literal (`all` is not blank).  The reference never consults the automaton for it:
// regex() answers with index(text, all) -- plain bytes, no framing, no decoding (forgex.F90:281-307).  Same sweep as
// above for the literal's first byte; a hit compares the whole literal; the smallest occurrence wins (64-bit atomicMin,
// key = S position of its first byte, so that the keys of several windows combine with MIN like any other start).
// An occurrence that would run past an open window end cannot be decided here: counted in best[1].
__global__ void __launch_bounds__(256) k_buffer_literal(const uint8_t* __restrict__ lit, int n, SparseParams sp, const uint8_t* __restrict__ buf,
                                                        ScanWindow W, unsigned long long* __restrict__ best) {
    const int lane = threadIdx.x & 31;
    const uint32_t FULL = 0xffffffffu;
    const int64_t len = W.len;
    const bool open_end = !W.last;
    const uintptr_t gbuf = reinterpret_cast<uintptr_t>(buf);
    const uintptr_t ubase = (gbuf + (uintptr_t)W.start_lo) & ~(uintptr_t)31;
    const int64_t nunits = W.start_hi > W.start_lo ? (int64_t)((gbuf + (uintptr_t)W.start_hi - ubase + 31) >> 5) : 0;
    const int64_t pos_base = (int64_t)ubase - (int64_t)gbuf;
    const int64_t gwarp = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5), nwarps = (int64_t)gridDim.x * 8;
    for (int64_t g0 = gwarp * 128; g0 < nunits; g0 += nwarps * 128) {
        unsigned long long cur = 0;
        if (lane == 0) cur = *reinterpret_cast<volatile unsigned long long*>(best);
        cur = __shfl_sync(FULL, cur, 0);
        if (cur != NO_START && (unsigned long long)(W.origin + pos_base + (g0 << 5)) + 2 > cur) break;   // behind the winner
        uint4 va[4], vb[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int64_t u = g0 + k * 32 + lane;
            va[k] = make_uint4(0, 0, 0, 0); vb[k] = va[k];
            if (u < nunits) {
                va[k] = ldg_nc_v4(reinterpret_cast<const void*>(ubase + ((uintptr_t)u << 5)));
                vb[k] = ldg_nc_v4(reinterpret_cast<const void*>(ubase + ((uintptr_t)u << 5) + 16));
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int64_t u = g0 + k * 32 + lane;
            if (u >= nunits) continue;
            const uint32_t w[8] = {va[k].x, va[k].y, va[k].z, va[k].w, vb[k].x, vb[k].y, vb[k].z, vb[k].w};
            uint32_t cand = 0;
#pragma unroll
            for (int q = 0; q < 8; q++) cand |= pack_byte_flags(first_mask<-1, false>(sp, w[q])) << (4 * q);
            const int64_t P = pos_base + (u << 5);
            if (P < W.start_lo) cand &= 0xFFFFFFFFu << (int)(W.start_lo - P);
            if (P + 32 > W.start_hi) cand &= (P >= W.start_hi) ? 0u : (0xFFFFFFFFu >> (int)(P + 32 - W.start_hi));
            while (cand) {                                     // ascending: the first occurrence of the unit ends the loop
                const int64_t pos = P + __ffs(cand) - 1;
                cand &= cand - 1;
                if (pos + n > len) { if (open_end) atomicAdd(best + 1, 1ull); break; }
                bool eq = true;
                for (int j = 0; j < n && eq; j++) eq = __ldg(buf + pos + j) == __ldg(lit + j);
                if (eq) { atomicMin(best, (unsigned long long)(W.origin + pos) + 2); break; }
            }
        }
    }
}

// A pattern whose prefix literal can overlap itself, or that has a suffix literal: the reference's candidate list is the
// NON-OVERLAPPING occurrences of the prefix, left to right, cut short by the last occurrence of the suffix
// (utility_m.f90:58-117, api_internal_m.F90:76-164) -- a sequential rule.  One thread replays it exactly as the batch
// kernels do for a string (eval_regex): always right, never fast (tens of MB/s); the parallel scans above serve every
// other pattern.
__global__ void k_buffer_sequential(KParams p, const uint8_t* __restrict__ buf, int64_t len, int64_t* __restrict__ from_to,
                                    const unsigned long long* __restrict__ pre_key, const unsigned long long* __restrict__ suf_key) {
    // Two parallel sweeps have looked for the prefix and the suffix literal (k_buffer_literal).  The prefix occurs and the
    // suffix occurs nowhere: the reference finds its first candidate, then index(text, suffix, back=.true.) == 0 ends the
    // search (api_internal_m.F90:94-102) -- no match, without walking anything (`a.*b` over a text without `b`).
    if (pre_key != nullptr && *pre_key != NO_START && *suf_key == NO_START) { from_to[0] = 0; from_to[1] = 0; return; }
    // The reference's loop is quadratic when candidates are many and attempts long (`aa.*[xy]` over a megabyte of `a`), and
    // for a sequential candidate list there is no linear-time stand-in: the replay stops after 16 byte steps per text byte
    // and reports (-2, -2) = FX_ERR_WORK_BUDGET instead of occupying the GPU for hours.
    long long steps = (long long)len * 16 + (4ll << 20);
    p.steps_left = &steps;
    Table<3> T;
    T.g_table = p.ctable; T.g_cmap = p.classmap; T.shift = p.c_row_shift; T.s_table = 0; T.s_cmap = 0;
    int64_t f, t;
    eval_regex(p, T, FetchGlobal{buf}, len, f, t);
    from_to[0] = f;
    from_to[1] = t;
}

// second step: longest end for the winning start; also the literal / degenerate cases.  `key` is the winning
// start as an S position of the whole text; the window must hold the text from that start to the end of its match.
__global__ void k_buffer_finish(KParams p, const uint8_t* __restrict__ buf, ScanWindow W,
                                const unsigned long long* __restrict__ best, int64_t* __restrict__ from_to, int whole_text,
                                const unsigned long long* __restrict__ done, const unsigned long long* __restrict__ use_alt,
                                const unsigned long long* __restrict__ best_alt, const unsigned long long* __restrict__ spent) {
    if (done != nullptr && *done != 0) return;              // the state-map scan has answered
    if (spent != nullptr && *spent != 0) { from_to[0] = -2; from_to[1] = -2; return; }   // a budgeted scan without a stand-in gave up
    if (use_alt != nullptr && *use_alt != 0) best = best_alt;   // the budgeted scan gave up and the state-map scan declined: the re-run's result
    Table<3> T;
    T.g_table = p.ctable; T.g_cmap = p.classmap; T.shift = p.c_row_shift; T.s_table = 0; T.s_cmap = 0;
    FetchGlobal fetch{buf};
    const int64_t len = W.len;
    int64_t from = 0, to = 0;
    if (p.all_active) {                                      // literal pattern: k_buffer_literal has found its first occurrence
        const unsigned long long key = *best;
        if (key != NO_START) { from = (int64_t)key - 1; to = from + p.all_len - 1; }
    } else if (whole_text && (len == 0 || (len == 1 && fetch(0) == 0x20))) {
        eval_regex(p, T, fetch, len, from, to);              // api_internal_m.F90:68-74 -> (0, 0)
    } else {
        const unsigned long long key = *best;
        const Anchored A{p.flags, p.start_nul, p.q0};
        if (key != NO_START) {
            const int64_t start = (int64_t)key - W.origin;      // S position relative to this window
            if (W.last) {
                const int64_t last = attempt_at(A, T, fetch, len, start);
                const int64_t f = start - 1 < 1 ? 1 : start - 1;
                const int64_t t = last < len ? last : len;
                if (f > 0 && t > 0) { from = W.origin + f; to = W.origin + t; }
            } else {
                // open window: walk the bytes we have; still alive at the window end -> the end is not known here
                uint32_t w = start == 1 ? (uint32_t)A.start_nul : (uint32_t)A.q0;
                int64_t seq = 0, last = (start == 1 && (__ldg(A.flags + A.start_nul) & SF_ACC)) ? 0 : -1;
                bool inter = false, alive = (w & W_STATE) != 0;
                for (int64_t j = start == 1 ? 0 : start - 2; alive && j < len; j++) {
                    const uint32_t c = fetch(j);
                    if (inter && (c & 0xC0) != 0x80) {
                        const uint32_t fl = __ldg(A.flags + (w & W_STATE));
                        for (int k = 1; k <= (int)(j - seq); k++) if (fl & (SF_FAILACC1 << (k - 1))) last = seq + k;
                        inter = false;
                    }
                    const uint32_t nw = T.next(w & W_STATE, c);
                    if ((nw & W_INTER) && !inter) seq = j;
                    inter = (nw & W_INTER) != 0;
                    w = nw;
                    if (w & W_ACC) last = j + 1;
                    alive = (w & W_STATE) != 0;
                }
                if (alive) { from = -1; to = -1; }          // undecided: the caller needs a longer window
                else {
                    const int64_t f = start - 1 < 1 ? 1 : start - 1;
                    if (f > 0 && last > 0) { from = W.origin + f; to = W.origin + last; }
                }
            }
        }
    }
    from_to[0] = from;
    from_to[1] = to;
}

// ---- NFA engine kernels: one thread per text (patterns past the eager state cap; correctness path, not a fast one) ----
template <int OP>
__device__ inline bool nfa_bool(const KParams& p, const NfaEngine& N, const uint8_t* __restrict__ s, int64_t len) {
    const uint8_t* pre = p.lits + p.all_len;
    const uint8_t* suf = pre + p.pre_len;
    FetchGlobal fetch{s};
    if (OP == 1) {
        if (p.all_active) return lit_index(s, len, p.lits, p.all_len) > 0;            // literal fast path (forgex.F90:111-130)
        if (len == 0 || (len == 1 && fetch(0) == 0x20)) return p.q0_accepting != 0;
        Anchored A{nullptr, 0, 0};
        int64_t f, t;
        including_exact(A, N, fetch, len, pre, p.pre_len, p.pre_active != 0, suf, p.suf_len, p.suf_active != 0, f, t);
        return f > 0 && t > 0;
    }
    if (p.all_active && len == p.all_len) return lit_equal(s, p.lits, p.all_len);     // forgex.F90:207-213
    // prefix / suffix gate of do_matching_exactly (api_internal_m.F90:199-233)
    const int64_t lp = p.pre_len, ls = p.suf_len;
    if (len > 0 && lp > 0 && lp == len && lit_equal(s, pre, (int)lp)) return true;
    if (lp > len || ls > len) return false;
    if (len > 0) {
        if (p.pre_active && !lit_equal(s, pre, (int)lp)) return false;
        if (p.suf_active && !lit_equal(s + (len - ls), suf, (int)ls)) return false;
    } else {
        if (p.pre_active && lp != 0) return false;
        if (p.suf_active && ls != 0) return false;
    }
    return nfa_match(N, fetch, len);
}
template <int OP>
__global__ void __launch_bounds__(64) k_nfa_bool(KParams p, NfaEngine N, const uint8_t* __restrict__ buf, const int64_t* __restrict__ offsets,
                                                 int64_t stride, int64_t n, uint8_t* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o0 = offsets ? __ldg(offsets + i) : i * stride, o1 = offsets ? __ldg(offsets + i + 1) : (i + 1) * stride;
        out[i] = nfa_bool<OP>(p, N, buf + o0, o1 - o0) ? 1 : 0;
    }
}
__global__ void __launch_bounds__(64) k_nfa_regex(KParams p, NfaEngine N, const uint8_t* __restrict__ buf, const int64_t* __restrict__ offsets,
                                                  int64_t n, int64_t single_len, int64_t* __restrict__ from, int64_t* __restrict__ to) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o0 = offsets ? __ldg(offsets + i) : 0, o1 = offsets ? __ldg(offsets + i + 1) : single_len;
        int64_t f, t;
        eval_regex(p, N, FetchGlobal{buf + o0}, o1 - o0, f, t);
        from[i] = f;
        to[i] = t;
    }
}

}  // namespace fxk
