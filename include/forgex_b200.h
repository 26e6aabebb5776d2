/* forgex_b200.h -- C ABI of the B200-native Forgex matching path.
 *
 * One shared library (forgex_b200/libforgex_b200.so) = host-side pattern compiler (C++) +
 * hand-written sm_100a kernels.  The entry points are what a `bind(C)` interface block in
 * Forgex's api_internal_m / forgex modules would bind (INTEGRATION.md shows the Fortran side):
 *
 *   reference interface                                   replaced by
 *   ----------------------------------------------------  ---------------------------------------
 *   do_matching_exactly    (src/api_internal_m.F90:171)    fx_match_fixed / fx_match_batch
 *   do_matching_including  (src/api_internal_m.F90:31)     fx_in_fixed / fx_in_batch,
 *                                                          fx_regex_batch / fx_regex_buffer
 *   automaton%preprocess + %init (src/automaton_m.F90:53-100,
 *     called per API call at src/forgex.F90:139-140)       fx_compile (once per pattern)
 *   operator(.in.)    (src/forgex.F90:74)                  fx_in        (one pattern, one text)
 *   operator(.match.) (src/forgex.F90:163)                 fx_match
 *   regex / regex_f   (src/forgex.F90:235, :351)           fx_regex
 *   is_valid_regex    (src/forgex.F90:58)                  fx_is_valid_regex
 *
 * Conventions
 *   - plain pointers and sizes only; byte strings are (pointer, int64 length), never NUL terminated.
 *   - every call returns an int status: 0 = ok; 1..24 = Forgex's own SYNTAX_* codes
 *     (src/essential/error_m.F90:12-38); 101.. = conditions listed below; negative = -(cudaError_t).
 *   - results are Forgex's: booleans as one byte (0/1) per string; spans as 1-based inclusive
 *     (from, to) in text coordinates, (0, 0) = no match, exactly what `regex` would return in its
 *     `from=` / `to=` arguments (src/forgex.F90:323-343).
 *   - `_dev` variants take DEVICE pointers and a cudaStream_t (as void*; NULL = default stream),
 *     enqueue asynchronously and copy nothing.  The variants without suffix take HOST pointers,
 *     copy in, run, copy out and return when the results are in host memory.
 *   - a compiled pattern is immutable after fx_compile; concurrent calls on distinct streams are safe.
 *   - there is no CPU fallback: without a usable CUDA device every matching call fails with
 *     FX_ERR_NO_DEVICE.  fx_compile and the fx_pattern_* queries are host-only.
 */
#ifndef FORGEX_B200_H
#define FORGEX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fx_pattern fx_pattern;

enum {               /* which entry point the pattern is compiled for (each has its own preprocessing
                        of the pattern text and its own automaton, src/forgex.F90:95, :182-190, :260) */
    FX_OP_MATCH = 0, /* .match.  */
    FX_OP_IN = 1,    /* .in.     */
    FX_OP_REGEX = 2  /* regex / regex_f (spans) */
};

enum {               /* where the transition table lives while a kernel runs */
    FX_TABLE_AUTO = 0,   /* shared memory when it fits, else global (L2-resident) */
    FX_TABLE_SMEM = 1,   /* force shared memory (error if it does not fit) */
    FX_TABLE_GLOBAL = 2  /* force the global / L2 path */
};

enum {
    FX_OK = 0,
    FX_ERR_TREE_NODE_LIMIT = 101,      /* Forgex `error stop`s here (src/ast/syntax_tree_graph_m.F90:115-117) */
    FX_ERR_DFA_STATE_CAP = 102,        /* eager construction exceeds 16383 states (Forgex's own ceiling for the
                                          lazily visited states: src/lazy_dfa/lazy_dfa_graph_m.F90:90-92) AND the NFA
                                          engine cannot take over (more than 8191 NFA states), or an entry point that
                                          needs the table engine was called on an NFA-engine handle; the linear-time
                                          window form (fx_statemap_*) also answers it for a pattern without the span
                                          path (fx_pattern_info.statemap == 0) */
    FX_ERR_PREFILTER_UNSUPPORTED = 103,/* WINDOW forms only (a text split across GPUs): the pattern's candidate list is
                                          sequential -- a prefix literal that can overlap itself, or a suffix literal
                                          (src/essential/utility_m.f90:58-117).  fx_regex_buffer* itself answers such
                                          patterns (one thread replays the reference's rule: exact, slow).  The
                                          linear-time window form (fx_statemap_*) answers it for every pattern with an
                                          extracted prefix literal and for literal-only patterns */
    FX_ERR_BAD_ARGUMENT = 104,
    FX_ERR_NO_DEVICE = 105,
    FX_ERR_WORK_BUDGET = 106           /* fx_regex_buffer* only: Forgex's own loop would need more than 16 byte steps per text
                                          byte on this text (many candidate starts, each running long) and the pattern has
                                          no linear-time stand-in (a sequential candidate list, or a prefix literal that is
                                          not provably a prefix of every match).  The reference would grind through it; the
                                          library stops instead.  The _dev forms report it as (from, to) = (-2, -2). */
};

typedef struct fx_pattern_info {
    int32_t op;
    int32_t status;
    int32_t nfa_states;
    int32_t cp_states;        /* states of the eager code-point automaton */
    int32_t cp_classes;
    int32_t byte_states;      /* states of the byte-level DFA (boundary + in-sequence states) */
    int32_t byte_classes;     /* byte equivalence classes */
    int32_t row_shift;        /* log2 of the padded row length of the class-compressed table */
    int32_t table_bytes;      /* class-compressed table size */
    int32_t direct_bytes;     /* 256-column table size */
    int32_t literal_all_len;  /* Forgex's extracted literals (src/ast/syntax_tree_optimize_m.F90:42) */
    int32_t literal_prefix_len;
    int32_t literal_suffix_len;
    int32_t literal_only;     /* 1: `all` is non-blank, the automaton is never consulted by .in./regex */
    int32_t residency;        /* FX_TABLE_* actually used by the last launch (0 before any launch) */
    int32_t direct;           /* 1: last launch used the 256-column table */
    int32_t prefix_mode;      /* `.in.` with an extracted prefix: 0 none, 1 prefilter is result-neutral for ASCII
                                 text (texts with bytes >= 0x80 are re-checked exactly), 2 always replayed exactly */
    int32_t sparse;           /* `.in.`: 1 when ragged batches run on the sparse-start kernel (the set F of first bytes
                                 that can begin a match is small) */
    int32_t sparse_ranges;    /* ASCII part of F as byte ranges [sparse_lo[i], sparse_hi[i]] */
    int32_t sparse_lo[4];
    int32_t sparse_hi[4];
    int32_t sparse_high;      /* 1: F also holds bytes >= 0xC0 (lead bytes; every such byte is tried as a start) */
    int32_t sparse_second;    /* >= 0: F is one byte and only this ASCII byte (or a lead byte) can follow it: the sweep
                                 tests for the byte pair; -1 otherwise */
    int32_t sparse_used;      /* 1: the last ragged `.in.` launch / buffer scan used the SWAR first-byte sweep */
    int32_t prefix_scan;      /* FX_OP_REGEX with an extracted prefix literal: 1 when the long-buffer path takes the literal's
                                 occurrences as candidates in parallel (the literal has no border and there is no suffix
                                 literal); 0: the candidate list is sequential -- fx_regex_buffer* replays it on one thread,
                                 the window forms answer FX_ERR_PREFILTER_UNSUPPORTED */
    int32_t statemap;         /* FX_OP_REGEX: 1 when the pattern has the linear-time span path (forward "ordered groups"
                                 automaton + reverse automaton): ragged batches run on it (K3f), and fx_regex_buffer* can
                                 fall back on the chunked state-map scan (K5) */
    int32_t nfa_engine;       /* 1: the eager automaton passes the state cap and the pattern is matched by NFA simulation on
                                 the device instead (one thread per text, the reference's own subset step on bit sets).
                                 Forgex builds its DFA lazily, so it answers such patterns (test/test_api/test_case_005.f90:
                                 76-108).  Correctness path, not a fast one; the window forms and the all-matches / count
                                 entry points answer FX_ERR_DFA_STATE_CAP for such a handle */
    int32_t compact_used;     /* last fixed-stride launch: 1 / 2 when a big boolean automaton ran on its ASCII-columns table
                                 from shared / global memory (K1c: at most 4 byte classes among the ASCII bytes, 8 bytes per
                                 state; strings with bytes >= 0x80 are decided by the full table), else 0 */
    int32_t statemap_used;    /* last fx_regex_buffer* call: 0 candidate-start scan only; 1 state-map scan; 2 candidate-start
                                 scan under a work budget with the state-map scan behind it (which of the two answered is
                                 decided on the device) */
    int32_t gated;            /* FX_OP_MATCH / FX_OP_IN: 1 when every string of a batch has to pass the wrapper's literal gates
                                 before (or instead of) the automaton walk -- a literal-only pattern; `.match.` with any
                                 non-empty prefix or suffix literal (do_matching_exactly compares lengths too, so a literal
                                 that is blank but not empty counts); `.in.` with a prefix prefilter that is not provably
                                 neutral.  0: the batch kernels walk the automaton directly */
} fx_pattern_info;

/* ---- host-only ------------------------------------------------------------------------- */
const char* fx_status_message(int status);

/* Compile `pattern` for one entry point.  Always returns a handle in *out (unless arguments are
 * bad); the return value is the pattern's status (0 or a SYNTAX_* / FX_ERR_* code). */
int fx_compile(const void* pattern, int64_t plen, int op, fx_pattern** out);
/* The Fortran-side compile route (SURVEY 8f-1; fortran/forgex_b200_tables_m.F90): the host has run Forgex's own front end
 * (tree%build, extract_literal) and explored the automaton eagerly -- a breadth-first search calling automaton%construct
 * (src/automaton_m.F90:333) for every state and one representative symbol of each alphabet segment -- and hands over the
 * ANCHORED code-point DFA: cuts[ncls + 1] ascending code points with cuts[0] = 0 (class c = [cuts[c], cuts[c+1] - 1]),
 * delta[nstates x ncls] with state 0 = dead, accept[nstates], q0 = the state before any symbol; plus the three literals.
 * Every automaton and table of the handle (search automaton of `.in.`, span path, byte-level tables) is derived from it.
 * For FX_OP_MATCH the DFA must be that of the pattern after operator__match's own preprocessing (src/forgex.F90:182-190). */
int fx_compile_from_dfa(int op, const int32_t* cuts, int32_t ncls, const int32_t* delta, int32_t nstates, const uint8_t* accept,
                        int32_t q0, const void* all, int64_t all_len, const void* prefix, int64_t prefix_len,
                        const void* suffix, int64_t suffix_len, fx_pattern** out);
/* the anchored code-point DFA of an FX_OP_REGEX handle, in exactly that form (tests / tools):
 * scalars = {states, classes, q0, state after the leading NUL} */
int fx_pattern_cp_automaton(const fx_pattern* p, const int32_t** cuts, const int32_t** delta, const uint8_t** accept, int32_t scalars[4]);
int fx_pattern_free(fx_pattern* p);
int fx_pattern_get_info(const fx_pattern* p, fx_pattern_info* info);
int fx_pattern_set_residency(fx_pattern* p, int residency);
/* copies of the extracted literals (buffers of at least the lengths reported by get_info) */
int fx_pattern_literals(const fx_pattern* p, void* all, void* prefix, void* suffix);
/* read-only views of the host copies of the device tables (for tests / tools):
 * table: byte_states << row_shift uint16 words; direct: byte_states * 256 words;
 * classmap: 256 bytes; flags: byte_states bytes; scalars: {start, start_nul, q0, matched, q0_accepting, result_threshold} */
int fx_pattern_tables(const fx_pattern* p, const uint16_t** table, const uint16_t** direct,
                      const uint8_t** classmap, const uint8_t** flags, int32_t scalars[6]);
/* FX_OP_REGEX patterns also carry a linear-time span path (tests / tools): the 256-column table of the forward
 * "ordered groups" automaton in its span word format (state | RA << 12 | INTER << 14 | ACC << 15, see fx_internal.hpp;
 * scalars = {states, start, start state accepts, 0}; endinfo: one byte per state), and the reverse automaton over
 * code-point classes (rdelta: rstates x rclasses words, bit 15 = the destination holds the NFA entry; rpage / rmixed:
 * two-level class map of the code points below U+10000, NULL when absent; cuts: classes+1 ascending code points;
 * rscalars = {states, classes, start, mixed pages}).  Returns 1 when the pattern has no such path. */
int fx_pattern_span_tables(const fx_pattern* p, const uint16_t** direct, const uint8_t** endinfo, int32_t scalars[4],
                           const uint16_t** rdelta, const uint8_t** rpage, const uint8_t** rmixed, const int32_t** cuts,
                           int32_t rscalars[4]);
/* the NFA engine's tables of a handle with fx_pattern_info.nfa_engine == 1 (tests / tools): trans[(s * classes + c) * words ..]
 * = epsilon-closed successor set of NFA state s on class c, q0 = closure of the entry, cuts: classes + 1 code points;
 * scalars = {NFA states, 64-bit words per set, classes, exit state, q0 accepting}.  Returns 1 for a table-engine handle. */
int fx_pattern_nfa_tables(const fx_pattern* p, const uint64_t** trans, const uint64_t** q0, const int32_t** cuts, int32_t scalars[5]);
int fx_is_valid_regex(const void* pattern, int64_t plen, int* status);
/* is_valid_regex over an array of patterns (it is `pure elemental` in the reference, src/forgex.F90:58-71): patterns as
 * one flat buffer + n+1 ascending offsets; valid[i] = 1/0, status[i] = the SYNTAX_* code of pattern i
 * (src/essential/error_m.F90:12-38).  Either output may be NULL.  Host-only. */
int fx_is_valid_regex_batch(const void* patterns, const int64_t* offsets, int64_t n, uint8_t* valid, int32_t* status);

/* ---- device-pointer entry points (asynchronous on `stream`) ---------------------------- */
int fx_match_fixed_dev(fx_pattern* p, const uint8_t* d_buf, int64_t n, int64_t stride, uint8_t* d_out, void* stream);
int fx_in_fixed_dev(fx_pattern* p, const uint8_t* d_buf, int64_t n, int64_t stride, uint8_t* d_out, void* stream);
/* offsets: n+1 ascending int64 byte offsets into d_buf; string i = d_buf[offsets[i] .. offsets[i+1]) */
int fx_match_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                       uint8_t* d_out, void* stream);
int fx_in_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                    uint8_t* d_out, void* stream);
int fx_regex_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                       int64_t* d_from, int64_t* d_to, void* stream);
/* one buffer of `len` bytes; d_from_to[0] = from, d_from_to[1] = to (64-bit, 1-based inclusive, 0/0 = none).
 * d_work: device scratch of fx_regex_buffer_work_bytes(len) bytes, 16-byte aligned (flags of the scans and the region
 * maps of the state-map scan; a few KB for small texts, at most 25 MB). */
int64_t fx_regex_buffer_work_bytes(int64_t len);
int fx_regex_buffer_dev(fx_pattern* p, const uint8_t* d_buf, int64_t len, int64_t* d_from_to, void* d_work, void* stream);

/* All matches, the way a caller of the reference collects them (README.md:197-222 shows the slicing): regex(), take
 * the match, regex() again on the rest text(to+1:), until nothing is found.  Stated semantics: every call frames ITS
 * text afresh (src/api_internal_m.F90:55) -- the rest begins behind a new leading NUL, so `^` matches at every restart
 * -- and the blank-text rule (src/api_internal_m.F90:68-74) applies to the rest; matches are never empty.
 * fx_regex_count_batch*: the number of matches per string of a ragged batch (d_counts[n]).
 * fx_regex_buffer_all*: one buffer; the first `capacity` spans in whole-buffer coordinates, *count (HOST memory in both
 * forms) = the number of matches (may exceed capacity).  The _dev form synchronises `stream` (per far match, or per
 * thousand near ones) and needs fx_regex_buffer_work_bytes(len) bytes of scratch.
 * fx_regex_all_batch*: every match of every string of a ragged batch, as CSR rows + flat spans.  rows[n + 1]: rows[0] = 0
 * and rows[i + 1] - rows[i] = the number of matches of string i (so rows[1..n] is the inclusive prefix sum of what
 * fx_regex_count_batch returns, and rows[n] is the total).  from[k], to[k] for k in [rows[i], rows[i + 1]) are string
 * i's matches in order, 1-based inclusive in the STRING's own coordinates (as fx_regex_batch returns them).  Only
 * indices k < capacity are written; rows is always complete, so a caller can read rows[n] and call again with room for
 * every span.  Every match advances the rest by at least one byte, so rows[n] <= total_bytes: a capacity of
 * total_bytes is always enough.  The _dev form is fully asynchronous (no host sync, nothing read back): the counts go
 * to d_rows + 1, d_rows[0] = 0 (also for n = 0), d_rows[1..n] is scanned in place, then the span pass runs -- not at
 * all for capacity 0, a cheap "rows only" call.  d_work: fx_regex_all_batch_work_bytes(n) bytes of device scratch,
 * 8-byte aligned (8 bytes per block of the scan, one block per 1024 strings up to 1024 blocks: at most 8 KB; computed
 * on the host).  Status codes are those of fx_regex_count_batch*. */
int fx_regex_count_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                             int64_t* d_counts, void* stream);
int fx_regex_buffer_all_dev(fx_pattern* p, const uint8_t* d_buf, int64_t len, int64_t* d_from, int64_t* d_to, int64_t capacity,
                            int64_t* count, void* d_work, void* stream);
int64_t fx_regex_all_batch_work_bytes(int64_t n);
int fx_regex_all_batch_dev(fx_pattern* p, const uint8_t* d_buf, const int64_t* d_offsets, int64_t n, int64_t total_bytes,
                           int64_t* d_rows, int64_t* d_from, int64_t* d_to, int64_t capacity, void* d_work, void* stream);

/* Window forms of the buffer search, for a text that is split across GPUs.  A window is a contiguous piece of the
 * text held by this GPU: window byte 0 is text position `origin` (0-based).  fx_buffer_scan_dev tries the starts
 * [start_lo, start_hi) of the window (attempts may read on to the end of the window) and lowers d_best[0] to the
 * smallest winning start, expressed as a 1-based position in NUL||text||NUL of the WHOLE text (so results of several
 * GPUs combine with a plain MIN); d_best[1] counts attempts that were still alive at an open window end (they could
 * not be decided: widen the halo).  A pattern with an extracted prefix literal (fx_pattern_info.prefix_scan) takes its
 * candidate starts from the literal's occurrences, as the reference does (src/api_internal_m.F90:76-104), and d_best[2]
 * becomes non-zero when the scanned starts hold an occurrence; when the literal occurs NOWHERE in the whole text the
 * reference tries every boundary instead: the caller then repeats the scan with fx_buffer_scan_all_dev.
 * The caller initialises d_best[0] = ~0, d_best[1] = d_best[2] = 0 (3 words).  is_first / is_last say
 * whether the window begins / ends where the text does.  Windows that do not begin the text need >= 3 bytes in
 * front of start_lo (character-boundary look-back).  fx_buffer_finish_dev turns a winning start (*d_key) into the
 * (from, to) span; it needs a window that holds the whole match, and answers (-1, -1) if the window ends first. */
int fx_buffer_scan_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t start_lo, int64_t start_hi,
                       int64_t origin, int is_first, int is_last, uint64_t* d_best, void* stream);
int fx_buffer_scan_all_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t start_lo, int64_t start_hi,
                           int64_t origin, int is_first, int is_last, uint64_t* d_best, void* stream);
int fx_buffer_finish_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t origin, int is_last,
                         const uint64_t* d_key, int64_t* d_from_to, void* stream);

/* Linear-time window form: the chunked state-map scan of fx_regex_buffer* over a text split across GPUs.  Each GPU
 * computes the SLAB MAP of its slab, the maps are gathered and combined (the same answer on every GPU), and a backward
 * walk finds the start of the match, handed from GPU to GPU when the match crosses slabs.  No attempt is replayed:
 * the work is linear in the text whatever the pattern, where the window scan above runs Forgex's own candidate loop.
 * Served: FX_OP_REGEX handles with the span path (fx_pattern_info.statemap) and no prefix literal; others get the codes
 * listed at FX_ERR_DFA_STATE_CAP and FX_ERR_PREFILTER_UNSUPPORTED.
 * fx_statemap_window_dev: the slab map of window bytes [slab_lo, slab_hi) (window byte 0 is text position `origin`).
 *   The window must hold min(64, origin + slab_lo) bytes in front of slab_lo (else FX_ERR_BAD_ARGUMENT); it needs no
 *   look-ahead.  d_map: FX_STATEMAP_MAP_WORDS int64 words = status (0 ok, 1 declined: more than 32 states can arrive at
 *   the slab, 2 empty slab = the identity), key count, 32 keys (states at the slab's start), 32 end states, 32 last
 *   accepts (text positions; -1 none, FX_STATEMAP_UNKNOWN: this key's walk could not be decided in the slab).
 *   d_work: fx_regex_buffer_work_bytes(slab_hi - slab_lo) bytes.
 * fx_statemap_combine (host-only): chains `nmaps` slab maps in text order from the start state, skipping empty slabs
 *   and stopping when the state dies, then takes the end-of-text step.  out[0] = end of the match (1-based `to`;
 *   text_len + 1 when the trailing NUL was consumed; <= 0 none), out[1] = 1 when the scan declined (a slab declined,
 *   or the true state met an unknown key): answer with the window scan instead.
 * fx_statemap_back_dev: advances the backward walk held in d_walk (FX_STATEMAP_WALK_WORDS int64 words = position,
 *   best start so far, reverse state, end of the match).  The caller starts it as {0, 0, FX_STATEMAP_WALK_NEW, out[0]}
 *   on the GPU that holds text byte end - 1 (the last GPU when end == text_len + 1).  The walk goes as far as the
 *   window allows; while d_walk[2] != FX_STATEMAP_WALK_DONE it continues on the GPU that holds byte d_walk[0] - 1
 *   (at most one hand-over per slab the match crosses).  When done, d_walk[0..1] = (from, to): exactly what
 *   fx_regex_buffer returns for the whole text. */
#define FX_STATEMAP_MAP_WORDS 98
#define FX_STATEMAP_UNKNOWN (-2)
#define FX_STATEMAP_WALK_WORDS 4
#define FX_STATEMAP_WALK_NEW (-1)
#define FX_STATEMAP_WALK_DONE (-2)
int fx_statemap_window_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t slab_lo, int64_t slab_hi,
                           int64_t origin, int64_t* d_map, void* d_work, void* stream);
int fx_statemap_combine(const fx_pattern* p, const int64_t* maps, int64_t nmaps, int64_t text_len, int64_t out[2]);
int fx_statemap_back_dev(fx_pattern* p, const uint8_t* d_window, int64_t window_len, int64_t origin, int64_t text_len,
                         int64_t* d_walk, void* stream);

/* ---- host-pointer entry points (copy in, run, copy out, synchronous) ------------------- */
int fx_match_fixed(fx_pattern* p, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out);
int fx_in_fixed(fx_pattern* p, const uint8_t* buf, int64_t n, int64_t stride, uint8_t* out);
int fx_match_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, uint8_t* out);
int fx_in_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, uint8_t* out);
int fx_regex_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, int64_t* from, int64_t* to);
int fx_regex_buffer(fx_pattern* p, const uint8_t* buf, int64_t len, int64_t* from, int64_t* to);
int fx_regex_count_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, int64_t* counts);
int fx_regex_buffer_all(fx_pattern* p, const uint8_t* buf, int64_t len, int64_t* from, int64_t* to, int64_t capacity, int64_t* count);
int fx_regex_all_batch(fx_pattern* p, const uint8_t* buf, const int64_t* offsets, int64_t n, int64_t* rows, int64_t* from,
                       int64_t* to, int64_t capacity);

/* ---- one pattern, one text: the reference's public API, compiled per call like the reference does */
int fx_in(const void* pattern, int64_t plen, const void* text, int64_t tlen, int* result);
int fx_match(const void* pattern, int64_t plen, const void* text, int64_t tlen, int* result);
/* regex(pattern, text, res, length, from, to, status): res = text(from:to).  Invalid pattern:
 * from = to = -9999, length = 0, *status = SYNTAX_* code, return value 0 (src/forgex.F90:266-274). */
int fx_regex(const void* pattern, int64_t plen, const void* text, int64_t tlen, int64_t* from, int64_t* to,
             int64_t* length, int* status);

/* The same three for `pure` Fortran callers (operator(.in.) / operator(.match.) are `pure elemental`, regex is a `pure
 * subroutine`, src/forgex.F90:24-54): a pure FUNCTION may only take intent(in) / value arguments, so the booleans come
 * back as the function value -- 1 / 0, or -status on failure -- and regex as a procedure without a result (*rc = status). */
int fx_in_value(const void* pattern, int64_t plen, const void* text, int64_t tlen);
int fx_match_value(const void* pattern, int64_t plen, const void* text, int64_t tlen);
void fx_regex_sub(const void* pattern, int64_t plen, const void* text, int64_t tlen, int64_t* from, int64_t* to, int64_t* length,
                  int* status, int* rc);

/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t fx_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* FORGEX_B200_H */
