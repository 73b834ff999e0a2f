// genztok.cu -- C ABI (include/genztok.h) and host orchestration of the CUDA pipeline.
//
// Per chunk of documents the device runs
//   k_cache_guard / k_cache_clear   make room in the word cache (reset when the worst case would not fit)
//   k_rows<G, FIXED>                split + cache lookup + framing + pad/truncate + mask + token types
//   k_bpe_pending                   BPE for the words that were new in this chunk
//   k_rows<G, FIXED> (row list)     redo the rows that met a new word
//   k_post_rows (row list)          rows with special ids inside the text (generic token types)
// and for ragged results (no padding / no truncation / max_len None or <= 0)
//   k_rows<COUNT> -> k_bpe_pending -> k_rows<COUNT> (row list) -> k_row_lens -> k_scan_i64
//   -> k_rows<RAGGED> -> k_post_rows.
// Long documents as windows (window.cuh): the ragged steps up to k_rows<RAGGED> per side -> k_window_count -> k_scan_i64
//   -> k_window_rows -> k_post_rows (row list).
// Pair truncation strategies (window.cuh): the ragged steps up to k_rows<RAGGED> per side -> k_window_rows<KEEP> (k_pair_rows)
//   -> k_post_rows<KEEP2> (row list).
// Decode is k_decode_len (lengths, trailing pad runs) -> k_scan_i64 -> k_decode_write.
// Extractive QA over the windows' offsets (qa.cuh): [k_qa_char_to_byte ->] k_qa_labels; k_qa_spans -> k_qa_spans_docs.
// MLM inputs and labels from an id plane (mlm.cuh): k_mlm_mask<WHOLE_WORD>.
// BPE-dropout rows (dropout.cuh): k_dropout_stream -> k_dropout_rows -> k_post_rows (row list); no word cache, no read-back.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/genztok.h"
#include "bpe.cuh"
#include "device_common.cuh"
#include "dropout.cuh"
#include "encode.cuh"
#include "flat.cuh"
#include "gather.cuh"
#include "host_tables.hpp"
#include "mlm.cuh"
#include "post.cuh"
#include "prep.cuh"
#include "qa.cuh"
#include "synth.cuh"
#include "window.cuh"

using namespace gzt;

namespace {

thread_local std::string g_create_err;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = n + n / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct ProfEvent { int name; cudaEvent_t a, b; int64_t alg; };

struct DeviceCtx {
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    size_t smem_optin = 0, smem_per_sm = 0;
    DevTables T{};
    WordCache C{};
    bool cache_ready = false;
    uint64_t cache_bytes = 0;                     // the chunk size the word cache is sized for
    bool cache_empty = true;                      // no word has been looked up since the cache was created or reset: the next text is all new
    bool force_wide = false;
    std::vector<void*> table_allocs;
    // chunk workspace
    DevBuf text, toff, pair, poff;                // inputs
    DevBuf ids, mask, tt, seq, row_len, seq_len, tt_len, status;   // outputs
    DevBuf L, keep, out_len, row_off, tail, redo, fix, misc, nwA, nwB, span_cnt, span_off, spans, scan_tmp, prep_out;
    DevBuf slots, key_arena, tok_arena, pending, ctr, rank_scratch;
    DevBuf len_arena;                             // piece byte lengths beside tok_arena (offset_mapping; allocated on first use)
    DevBuf offs;                                  // ragged pass: [total][2] token byte offsets (offset_mapping)
    DevBuf qa_ans, qa_win;                        // QA: byte spans converted from characters; per-window best spans
    const uint32_t* mlm_cont = nullptr;           // MLM (mlm.cuh): the handle's continuation bitset and replacement ids, uploaded
    const int32_t* mlm_repl = nullptr;            // on the first MLM call of this device
    DevBuf dec_lead;                              // decode: per-row description left by the length pass for the write pass
    DevBuf dec_stat;                              // decode, fixed-width rows: ids in front of the pad runs, summed by the length pass
    double dec_avg_lead = -1;                     // ... per row, once the host has read it (-1: not known for the current batch)
    DevBuf tok_flag, tok_len, tok_pos;            // decode of ragged rows by id: last-of-row flags, bytes per id, their scan
    int64_t tok_base = 0, tok_n = -1;             // the ids that scan describes
    struct { const void *ids = nullptr, *ids_off = nullptr, *out_off = nullptr; int64_t n = -1; int32_t width = 0; int by_id = 0; } dec_sig;   // the batch it describes
    struct FlatBufs { DevBuf dsb, st, tpref, cnt, wtok; } flat[2];   // byte-parallel pipeline, per side
    // host path, fixed layout: two sets of chunk buffers so that the copy of chunk i + 1 to the device, the kernels of chunk i and
    // the copy of chunk i - 1 to the host overlap (PCIe is full duplex); one stream each
    struct Stage {
        DevBuf text, toff, pair, poff, ids, mask, tt, seq, row_len, seq_len, status, extent;
        cudaEvent_t h2d = nullptr, k = nullptr, d2h = nullptr;
    } stage[2];
    cudaStream_t s_in = nullptr, s_out = nullptr;
    int32_t* h_extent = nullptr;                  // pinned: [2] staged-column extents of the two chunks in flight
    // byte-parallel pipeline: rows of more than 32 tokens in the last sampled call (k_flat_rows counts them; read back without a
    // synchronisation).  When hardly any row needs more, the next call stages 32 columns instead of 64 and leaves the rest to the pad boxes.
    unsigned long long* h_over32 = nullptr;       // pinned
    cudaEvent_t over32_ev = nullptr;
    bool over32_pending = false, stage32 = false;
    int64_t over32_rows = 0;
    // the shared work areas (word cache, lists, flat arrays) are used by one stream at a time: a call on another stream
    // first waits for the event the previous call left behind
    cudaEvent_t last_done = nullptr;
    cudaStream_t last_stream = nullptr;
    bool last_valid = false;
    // synthetic workload generator (synth.cuh): tables and the length scratch
    SynthTables synth{};
    bool synth_ready = false;
    DevBuf synth_len;
    // long documents as windows (window.cuh): token streams of the two sides, windows per document, the k_post_rows row list; the
    // batch step 1 of genztok_encode_windows_device described, for its step 2
    struct WinState {
        DevBuf ids[2], off[2], count, woff, fix, doc, start;
        DevBuf offs[2], plane_offs;               // offset_mapping: the streams' token offsets, and the host form's [K, W, 2] plane
        DevBuf len[2];                            // BPE-dropout: ids per slot of the capped streams (which live in ids[2])
        DevBuf drop_scratch, drop_keys;           // BPE-dropout: symbols and ranks of long words; the host form's row keys of a chunk
        struct { const void *a = nullptr, *a_off = nullptr, *b = nullptr, *b_off = nullptr, *win_off = nullptr; int64_t n = -1, a_bytes = 0, b_bytes = 0;
                 int32_t W = 0, s = 0; bool offs = false; } sig;
        int64_t n_win = -1;                       // windows of that batch; -1: no step 1 to continue from
    } win;
    // profiling
    bool profiling = false;
    std::vector<ProfEvent> events;
    std::vector<cudaEvent_t> free_events;
};

}  // namespace

struct genztok {
    HostTables H;
    std::vector<DeviceCtx*> devs;
    std::string err;
    std::atomic<int64_t> launches{0};
    std::mutex mu;                       // encode/decode calls are serialised per handle
    std::mutex err_mu;                   // guards err / prof_names (device worker threads)
    // options
    int64_t max_chunk_bytes = 64ll << 20;
    int64_t fixed_cache = 0;             // size the word cache for max_chunk_bytes at once instead of by the chunks met (test knob)
    int64_t chunk_rows = 1ll << 18;     // rows per chunk of the host path: small enough that the copies of neighbouring chunks overlap the kernels
    int64_t force_group = 0;
    int64_t force_wide = 0;              // stage rows as int32 even when ids fit uint16 (test knob)
    int64_t grid_mult = 1;               // row-kernel grid = resident blocks x grid_mult
    int64_t no_flat = 0;                 // use the fused row kernel even where the byte-parallel pipeline applies (test knob)
    int64_t no_stage32 = 0;              // byte-parallel pipeline: never narrow the staged columns to 32 by the previous call's row lengths (test knob)
    int64_t no_discovery = 0;            // fused row kernel on an empty cache: do not run the byte-parallel word pass first (test knob)
    int64_t flat_rows = 32;              // rows per warp tile of k_flat_rows
    int64_t no_side_pads = 0;            // k_flat_rows writes the pad columns itself (test knob)
    int64_t pad_box_cols = 0;            // columns per TMA pad box of the byte-parallel pipeline (multiple of 16; 0 = as wide as possible, up to 256)
    int64_t decode_write = 0;            // fixed-width decode, write pass: 0 = by the average lead, 1 = warp per row, 2 / 3 = lane per junction with 256 / 512 bytes (test knob)
    int64_t decode_wide_max = 64;        // average lead (ids) up to which the 512-byte junction kernel is taken (<= 14: never)
    int64_t no_copy_kernel = 0;          // host path: trimmed planes go back through cudaMemcpy2DAsync instead of k_copy_out (test knob)
    int64_t copy_blocks = 64;            // blocks of k_copy_out
    int64_t copy_round = 64;             // columns the one-byte planes' copy-out is rounded up to (32 or 64: whole 64-byte lines of host memory)
    int64_t l2_policy = 2;               // k_flat_words: bit 0: text read evict-first (slower), bit 1: word arrays stored evict-last (default: -3.5 % per chunk)
    int64_t rows_pad_pct = 0;            // share of the pad columns (percent of the 32-row tiles, the last ones) that k_flat_rows stores instead of k_flat_words
    int64_t rows_grid = 0;               // cap on resident blocks per SM of k_flat_rows (0 = as many as fit)
    int64_t rows_minb = 0, words_minb = 3;   // resident 256-thread blocks per SM the flat kernels are compiled for (rows: 0 = 3 for pairs, 5 for single sentences)
    int64_t no_tma = 0;                  // write the fixed planes with store instructions instead of the TMA unit (test knob)
    int64_t no_token_decode = 0;         // decode ragged rows with a warp per row instead of a thread per id (test knob)
    int64_t no_fixed_decode = 0;         // decode fixed-width rows with the any-rows kernels (test knob)
    int64_t force_kr = 0;                // staged columns per row of the TMA write-out (test knob; 0 = from the text size)
    std::vector<std::string> prof_names;
    struct ProfAcc { int64_t launches = 0; double ms = 0; int64_t alg = 0; };
    std::map<std::string, ProfAcc> prof_acc;
    // pinned host pool
    std::multimap<size_t, void*> host_pool;
    size_t host_pool_bytes = 0;
    std::mutex pool_mu;                  // guards host_pool (the device worker threads of a call take staging buffers from it)
    // What a pooled result plane still holds from its last use: the same [rows, width] shape with everything behind column
    // `dirty_cols` equal to padding.  A call that reuses it copies only the columns that can differ (see encode_fixed_pipelined).
    struct PlaneMeta { int64_t rows; int32_t width, dirty_cols, elt; int32_t pad; };
    std::map<void*, PlaneMeta> plane_meta;
    // MLM masking (mlm.cuh), built from the tables on the first MLM call: bit id of mlm_cont is set when decoder[id] ends in "@@";
    // mlm_repl lists, ascending, the ids in the decoder that are not special
    bool mlm_built = false;
    std::vector<uint32_t> mlm_cont;
    std::vector<int32_t> mlm_repl;
};

namespace {

int fail(genztok_t* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) { std::lock_guard<std::mutex> l(h->err_mu); h->err = buf; } else g_create_err = buf;
    return code;
}

#define CU(call)                                                                                           \
    do {                                                                                                   \
        cudaError_t _e = (call);                                                                           \
        if (_e != cudaSuccess) return fail(h, GENZTOK_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

int prof_name_id(genztok_t* h, const char* name) {
    std::lock_guard<std::mutex> l(h->err_mu);
    for (size_t i = 0; i < h->prof_names.size(); i++) if (h->prof_names[i] == name) return (int)i;
    h->prof_names.push_back(name);
    return (int)h->prof_names.size() - 1;
}

struct LaunchScope {   // counts the launch and, when profiling, brackets it with events on the stream
    genztok_t* h; DeviceCtx* d; ProfEvent ev{}; bool on;
    // alg_bytes: the algorithmic bytes of this launch (SURVEY.md 8 d4 split by kernel), reported next to its time
    LaunchScope(genztok_t* h_, DeviceCtx* d_, const char* name, int64_t alg_bytes = 0) : h(h_), d(d_), on(d_->profiling) {
        h->launches++;
        dbg_name = name;
        if (on) {
            ev.name = prof_name_id(h, name);
            ev.alg = alg_bytes;
            for (cudaEvent_t* e : {&ev.a, &ev.b}) {
                if (!d->free_events.empty()) { *e = d->free_events.back(); d->free_events.pop_back(); }
                else cudaEventCreate(e);
            }
            cudaEventRecord(ev.a, cur_stream);
        }
    }
    ~LaunchScope() {
        if (on) { cudaEventRecord(ev.b, cur_stream); d->events.push_back(ev); }
        static const bool debug = getenv("GENZTOK_DEBUG") != nullptr;
        if (debug) {   // serialise and name every launch (hang / fault localisation)
            cudaError_t e = cudaStreamSynchronize(cur_stream);
            fprintf(stderr, "[genztok] %s: %s\n", dbg_name, cudaGetErrorString(e));
            fflush(stderr);
        }
    }
    const char* dbg_name = "";
    static thread_local cudaStream_t cur_stream;
};
thread_local cudaStream_t LaunchScope::cur_stream = nullptr;

// Launch with the programmatic-stream-serialization attribute (see pdl_wait in device_common.cuh): the kernel may be scheduled
// while its predecessor in the stream drains, which takes most of the launch gap out of chains of short kernels.
template <class... KArgs, class... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

template <class T>
cudaError_t upload(DeviceCtx* d, const std::vector<T>& v, const T** out) {
    void* p = nullptr;
    size_t bytes = std::max<size_t>(v.size() * sizeof(T), 16);
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    d->table_allocs.push_back(p);
    if (!v.empty()) e = cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    *out = reinterpret_cast<const T*>(p);
    return e;
}

int init_device(genztok_t* h, DeviceCtx* d) {
    CU(cudaSetDevice(d->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, d->device));
    d->sm_count = prop.multiProcessorCount;
    d->smem_optin = prop.sharedMemPerBlockOptin;
    d->smem_per_sm = prop.sharedMemPerMultiprocessor;
    CU(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
    const HostTables& H = h->H;
    DevTables& T = d->T;
    CU(upload(d, H.pair_slots, &T.pair));
    T.pair_mask = H.pair_mask;
    CU(upload(d, H.cp_slots, &T.cp));
    T.cp_mask = H.cp_mask;
    CU(upload(d, H.id_cont, &T.id_cont));
    CU(upload(d, H.id_fin, &T.id_fin));
    CU(upload(d, H.sym_ncp, &T.sym_ncp));
    CU(upload(d, H.form_blob, &T.form_blob));
    CU(upload(d, H.mid_off, &T.mid_off));
    CU(upload(d, H.mid_len, &T.mid_len));
    CU(upload(d, H.last_off, &T.last_off));
    CU(upload(d, H.last_len, &T.last_len));
    CU(upload(d, H.mid_desc, &T.mid_desc));
    CU(upload(d, H.last_desc, &T.last_desc));
    { const HostTables::FastForm* ff = nullptr; CU(upload(d, H.mid_fast, &ff)); T.mid_fast = reinterpret_cast<const uint4*>(ff); }
    T.n_ids = (int32_t)H.n_ids;
    T.pad = H.special_id[0]; T.bos = H.special_id[1]; T.eos = H.special_id[2]; T.msk = H.special_id[3]; T.unk = H.special_id[4];
    T.specials_distinct = (T.pad != T.bos && T.pad != T.eos && T.bos != T.eos) ? 1 : 0;
    return GENZTOK_OK;
}

// Calls that use the device context's shared work areas on different streams are ordered by an event (the word cache, the
// redo / fix lists and the flat arrays belong to one call at a time).
int stream_enter(genztok_t* h, DeviceCtx* d, cudaStream_t st) {
    if (d->last_valid && d->last_stream != st) CU(cudaStreamWaitEvent(st, d->last_done, 0));
    return GENZTOK_OK;
}
int stream_leave(genztok_t* h, DeviceCtx* d, cudaStream_t st) {
    if (!d->last_done) CU(cudaEventCreateWithFlags(&d->last_done, cudaEventDisableTiming));
    CU(cudaEventRecord(d->last_done, st));
    d->last_stream = st; d->last_valid = true;
    return GENZTOK_OK;
}

int launch_guard(genztok_t* h, DeviceCtx* d, cudaStream_t st, int64_t chunk_bytes, int force, uint32_t* z0 = nullptr, uint64_t n0 = 0, uint32_t* z1 = nullptr,
                 uint64_t n1 = 0);

uint64_t next_pow2(uint64_t x) { uint64_t p = 1; while (p < x) p <<= 1; return p; }

// The word cache is sized for the worst case of ONE chunk (every second byte a new word), so its size follows the largest chunk this
// device has met (a power of two from 1 MiB up, at most max_chunk_bytes): a handle that only sees small batches keeps a 32 MiB table
// instead of the 2 GiB that max_chunk_bytes = 64 MiB would cost.  A larger chunk regrows it (and empties it).
int ensure_cache(genztok_t* h, DeviceCtx* d, cudaStream_t st, int64_t chunk_bytes) {
    const uint64_t limit = (uint64_t)h->max_chunk_bytes;
    const uint64_t need = std::min<uint64_t>(limit, (uint64_t)std::max<int64_t>(chunk_bytes, 0) + 64);
    if (d->cache_ready && need <= d->cache_bytes) return GENZTOK_OK;
    const uint64_t B = h->fixed_cache ? limit : std::min<uint64_t>(limit, std::max<uint64_t>(next_pow2(need), 1ull << 20));
    const uint64_t slots = std::max<uint64_t>(next_pow2(B), 1024);
    const bool regrow = d->cache_ready;
    if (regrow) CU(cudaDeviceSynchronize());                       // nothing may still be using the arrays that are about to be freed
    CU(d->slots.ensure(slots * sizeof(Slot)));
    CU(d->key_arena.ensure(B + B / 3 + 128));                      // (long keys are stored 8-byte aligned: up to 7 bytes of padding for 25 or more)
    CU(d->tok_arena.ensure((2 * B + 64) * 4));
    CU(d->pending.ensure((B / 2 + 64) * 4));
    CU(d->ctr.ensure(C_COUNT * 8));
    CU(d->rank_scratch.ensure((B + 64) * 4));
    // on the stream that runs the kernels of this call (the handle's own stream is non-blocking: nothing else orders it with the caller's)
    CU(cudaMemsetAsync(d->slots.p, 0, slots * sizeof(Slot), st));
    if (!regrow) CU(cudaMemsetAsync(d->ctr.p, 0, C_COUNT * 8, st));
    else {                                                           // keep the cumulative counters (errors, tokens)
        CU(cudaMemsetAsync(d->ctr.p, 0, (size_t)C_ERR * 8, st));
        CU(cudaMemsetAsync(d->ctr.as<unsigned long long>() + C_TOKENS + 1, 0, (size_t)(C_COUNT - C_TOKENS - 1) * 8, st));
    }
    WordCache& C = d->C;
    C.slots = d->slots.as<Slot>(); C.mask = (uint32_t)(slots - 1);
    C.key_arena = d->key_arena.as<uint8_t>(); C.key_cap = B + B / 3 + 64;
    C.tok_arena = d->tok_arena.as<uint32_t>(); C.tok_cap = 2 * B + 64;
    C.pending = d->pending.as<uint32_t>(); C.pending_cap = B / 2 + 64;
    C.ctr = d->ctr.as<unsigned long long>();
    C.rank_scratch = d->rank_scratch.as<uint32_t>(); C.rank_cap = B + 64;
    if (d->len_arena.p) CU(d->len_arena.ensure((2 * B + 64) * 2));
    d->cache_ready = true;
    d->cache_empty = true;
    d->cache_bytes = B;
    return GENZTOK_OK;
}

// offset_mapping needs the byte length of every piece of every cached word (k_bpe_pending records them once len_arena is
// allocated).  The first call on a device that asks for offsets allocates the lengths and empties the cache, so that every word
// cached from then on has them; a handle that never asks allocates nothing.  Call after ensure_cache.
int ensure_piece_lens(genztok_t* h, DeviceCtx* d, cudaStream_t st) {
    if (d->len_arena.p) return GENZTOK_OK;
    CU(d->len_arena.ensure((size_t)d->C.tok_cap * 2));
    int rc = launch_guard(h, d, st, 0, 1);
    if (rc) return rc;
    d->cache_empty = true;
    return GENZTOK_OK;
}

// Rows are staged in shared memory as uint16 when every vocabulary id fits (the bundled model: 48,423 ids).
bool narrow_ids(const DeviceCtx* d) { return !d->force_wide && d->T.n_ids <= 65536 && d->T.unk < 65536 && d->T.unk >= 0; }
size_t row_stage_bytes(const DeviceCtx* d, int32_t W, int D) {
    const size_t Wp = ((size_t)W + 3) & ~(size_t)3;
    return ((size_t)D * Wp * (narrow_ids(d) ? 2 : 4) + 15) & ~(size_t)15;
}

// Documents per warp tile: aim at ~26 sixteen-byte pieces of text per window, bounded by the shared memory
// the staged rows need (MODE_FIXED) so that four 8-warp blocks fit an SM when possible.
int pick_tile_docs(genztok_t* h, const DeviceCtx* d, int64_t bytes_a, int64_t bytes_b, int64_t n, int32_t W, bool fixed) {
    int D;
    if (h->force_group) D = (int)h->force_group;
    else {
        const int64_t avg = n > 0 ? std::max<int64_t>(std::max(bytes_a, bytes_b) / n, 1) : 1;
        D = (int)std::min<int64_t>(32, std::max<int64_t>(1, 416 / avg));
    }
    if (fixed) while (D > 1 && 8 * (sizeof(TileSmem) + row_stage_bytes(d, W, D)) > d->smem_optin / 2) D--;
    return D;
}

template <int MODE, typename TokT, bool TMA, bool OFFS = false>
int launch_rows_t(genztok_t* h, DeviceCtx* d, const RowArgs& A, cudaStream_t st, const char* name, int64_t n_items_hint, const TmaPlanes* M) {
    const int D = A.row_list ? 1 : A.D;
    auto smem_for = [&](int w) {
        if (TMA) return (M->PB ? tma_const_bytes(A.D, M->PB) : 0) + (size_t)w * (r128(sizeof(TileSmem)) + 2 * tma_stage_bytes(A.D, M->KR, A.has_pair && A.tt));
        return (size_t)w * (sizeof(TileSmem) + (MODE == MODE_FIXED ? row_stage_bytes(d, A.W, A.D) : 0));
    };
    int wpb = 8;
    while (wpb > 1 && smem_for(wpb) > d->smem_optin) wpb >>= 1;
    const size_t smem = smem_for(wpb);
    if (smem > d->smem_optin) return fail(h, GENZTOK_E_LIMIT, "row of %d ids does not fit shared memory", A.W);
    auto kern = k_rows<MODE, TokT, TMA, OFFS>;
    if (smem > 48 * 1024) CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 1;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, wpb * 32, smem));
    if (occ < 1) occ = 1;
    const int64_t tiles = (n_items_hint + D - 1) / D;
    int64_t blocks = std::min<int64_t>((tiles + wpb - 1) / wpb, (int64_t)d->sm_count * occ * h->grid_mult);
    if (blocks < 1) blocks = 1;
    static const TmaPlanes no_planes{};
    LaunchScope ls(h, d, name);
    CU(launch_pdl(kern, dim3((unsigned)blocks), dim3(wpb * 32), smem, st, d->T, d->C, A, TMA ? *M : no_planes));
    CU(cudaGetLastError());
    return GENZTOK_OK;
}
template <int MODE>
int launch_rows(genztok_t* h, DeviceCtx* d, const RowArgs& A, cudaStream_t st, const char* name, int64_t n_items_hint, const TmaPlanes* M = nullptr) {
    if (MODE == MODE_FIXED && M) return launch_rows_t<MODE_FIXED, int32_t, true>(h, d, A, st, name, n_items_hint, M);
    if (MODE == MODE_FIXED && narrow_ids(d)) return launch_rows_t<MODE, uint16_t, false>(h, d, A, st, name, n_items_hint, nullptr);
    if (MODE == MODE_RAGGED && A.offs) return launch_rows_t<MODE_RAGGED, int32_t, false, true>(h, d, A, st, name, n_items_hint, nullptr);
    return launch_rows_t<MODE, int32_t, false>(h, d, A, st, name, n_items_hint, nullptr);
}

// ---- TMA write-out set-up (see TmaPlanes in encode.cuh) -------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) { cudaGetLastError(); p = nullptr; }
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
// map of a row-major [n, W] plane with boxes of [rows x cols] elements
bool plane_map(CUtensorMap* m, void* base, int elt_bytes, int64_t n, int32_t W, int cols, int rows) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)W, (cuuint64_t)n};
    const cuuint64_t strides[1] = {(cuuint64_t)W * (cuuint64_t)elt_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)cols, (cuuint32_t)rows};
    const cuuint32_t estr[2] = {1, 1};
    return enc(m, elt_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_INT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// Decide whether this launch can use the TMA write-out and describe the planes.  KR (staged columns) follows the
// average text per row: ~3 bytes per token plus framing, at least 32; rows that need more take the generic second pass.
bool setup_tma(genztok_t* h, const DeviceCtx* d, const RowArgs& A, int64_t bytes, TmaPlanes* M, size_t tile_bytes = sizeof(TileSmem)) {
    if (h->no_tma || A.row_list || !A.ids || !A.mask || A.seq || A.n_rows < 1 || A.n_rows >= (1ll << 31)) return false;
    const int32_t W = A.W;
    if (W < 16 || (W & 15)) return false;
    auto misaligned = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) != 0; };
    if (misaligned(A.ids) || misaligned(A.mask) || (A.has_pair && A.tt && misaligned(A.tt))) return false;
    int64_t KR = h->force_kr;
    if (KR <= 0) KR = std::max<int64_t>(32, (bytes / A.n_rows / 3 + 12 + (A.has_pair ? 4 : 0) + 15) & ~15ll);
    if (KR + 16 > W) KR = W;
    if (KR > 256) return false;
    // columns per pad box: the constant buffer a block keeps for it costs shared memory (hence L1) in proportion
    int32_t PB = (int32_t)std::min<int64_t>(W - KR, 256);
    if (tile_bytes != sizeof(TileSmem) && h->pad_box_cols > 0 && PB > h->pad_box_cols)
        for (int32_t pb = (int32_t)h->pad_box_cols; pb >= 16; pb -= 16) if ((W - KR) % pb == 0) { PB = pb; break; }   // the widest box that tiles the pad columns
    const bool tt = A.has_pair && A.tt;
    if (tt && A.pad_i8 != 0) return false;      // the constant pad boxes of token_type_ids are zeros: a pad id that is not 0 takes the store path
    if (tile_bytes == sizeof(TileSmem)) {
        // the fused kernel is latency bound: the staging must not cost occupancy (four 8-warp blocks per SM), else the store path wins
        if (!h->force_kr && 4 * ((PB ? tma_const_bytes(A.D, PB) : 0) + 8 * (r128(tile_bytes) + 2 * tma_stage_bytes(A.D, (int)KR, tt)) + 1024) > d->smem_per_sm) return false;
        if (2 * ((PB ? tma_const_bytes(A.D, PB) : 0) + 8 * (r128(tile_bytes) + 2 * tma_stage_bytes(A.D, (int)KR, tt)) + 1024) > d->smem_optin) return false;
    } else {
        // k_flat_rows: the constant pad boxes and one row buffer per warp
        if (2 * ((PB ? tma_const_bytes(A.D, PB) : 0) + 8 * (r128(tile_bytes) + r128((size_t)KR * 4)) + 1024) > d->smem_optin) return false;
    }
    memset(M, 0, sizeof *M);
    M->KR = (int32_t)KR; M->PB = PB;
    bool ok = plane_map(&M->ids_real, A.ids, 4, A.n_rows, W, (int)KR, A.D) && plane_map(&M->mask_real, A.mask, 1, A.n_rows, W, (int)KR, A.D);
    if (ok && tt) ok = plane_map(&M->tt_real, A.tt, 1, A.n_rows, W, (int)KR, A.D);
    if (ok && PB) {
        ok = plane_map(&M->ids_pad, A.ids, 4, A.n_rows, W, PB, A.D) && plane_map(&M->mask_pad, A.mask, 1, A.n_rows, W, PB, A.D);
        if (ok && tt) ok = plane_map(&M->tt_pad, A.tt, 1, A.n_rows, W, PB, A.D);
    }
    return ok;
}

// Can the fixed-layout kernel stage one row of W ids (one document per tile, one warp per block)?
bool fixed_fits(const DeviceCtx* d, int32_t W) { return sizeof(TileSmem) + row_stage_bytes(d, W, 1) <= d->smem_optin; }

int launch_guard(genztok_t* h, DeviceCtx* d, cudaStream_t st, int64_t chunk_bytes, int force, uint32_t* z0, uint64_t n0, uint32_t* z1, uint64_t n1) {
    {
        LaunchScope ls(h, d, "k_cache_guard");
        CU(launch_pdl(k_cache_guard, dim3(1), dim3(1), 0, st, d->C, (unsigned long long)(chunk_bytes / 2 + 2), (unsigned long long)(chunk_bytes + chunk_bytes / 3 + 8), (unsigned long long)(chunk_bytes + chunk_bytes / 2 + 2), force));
    }
    {
        LaunchScope ls(h, d, "k_cache_clear");
        CU(launch_pdl(k_cache_clear, dim3(d->sm_count * 4), dim3(256), 0, st, d->C, z0, n0, z1, n1));
    }
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

int launch_bpe(genztok_t* h, DeviceCtx* d, cudaStream_t st) {
    LaunchScope ls(h, d, "k_bpe_pending");
    CU(launch_pdl(k_bpe_pending, dim3(d->sm_count * 6), dim3(256), 0, st, d->T, d->C, d->len_arena.as<uint16_t>()));      // latency bound (pair-table look-ups): as many warps as fit
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

// out[0..n] = exclusive scan of in[0..n): one block for small inputs, tiles + totals + fix-up otherwise
int launch_scan(genztok_t* h, DeviceCtx* d, cudaStream_t st, const int64_t* in, int64_t* out, int64_t n) {
    if (n <= 2 * SCAN_TILE) {
        LaunchScope ls(h, d, "k_scan_i64");
        k_scan_i64<<<1, 1024, 0, st>>>(in, out, n);
        CU(cudaGetLastError());
        return GENZTOK_OK;
    }
    const int64_t nt = (n + SCAN_TILE - 1) / SCAN_TILE;
    CU(d->scan_tmp.ensure((size_t)(2 * nt + 2) * 8));
    int64_t* tsum = d->scan_tmp.as<int64_t>();
    int64_t* texcl = tsum + nt;
    { LaunchScope ls(h, d, "k_scan_tiles"); k_scan_tiles<<<(unsigned)nt, 1024, 0, st>>>(in, out, tsum, n); }
    { LaunchScope ls(h, d, "k_scan_i64"); k_scan_i64<<<1, 1024, 0, st>>>(tsum, texcl, nt); }
    { LaunchScope ls(h, d, "k_scan_fix"); k_scan_fix<<<(unsigned)nt, 1024, 0, st>>>(out, texcl, n, nt); }
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

int8_t pad_as_i8(const DeviceCtx* d) { return (d->T.pad >= 0 && d->T.pad <= 127) ? (int8_t)d->T.pad : (int8_t)GENZTOK_PAD_MARK; }
int8_t eos_as_i8(const DeviceCtx* d) { return (d->T.eos >= 0 && d->T.eos <= 127) ? (int8_t)d->T.eos : (int8_t)GENZTOK_EOS_MARK; }

// work arrays of the byte-parallel pipeline for one side (flat.cuh)
uint64_t flat_chunks(int64_t nbytes) {
    const uint64_t nG = (((uint64_t)nbytes + 15) >> 5) + 3;                 // granules (+ slack for the clamp in flat_hi)
    return (nG + FC_OWN - 1) / FC_OWN + 1;                                   // chunks
}
// (the word arrays of both sides are one allocation, side B's behind side A's: k_flat_rows addresses them with one base pointer)
int flat_side_setup(genztok_t* h, DeviceCtx* d, int s, const Side& side, const Side* other, int64_t n, FlatSide* out) {
    DeviceCtx::FlatBufs& B = d->flat[s];
    const uint64_t nB = flat_chunks(side.nbytes);
    const uint64_t ng = nB * FC_OWN + 2;
    CU(B.dsb.ensure(ng * 4)); CU(B.st.ensure(ng * 4)); CU(B.tpref.ensure(ng * 2));
    CU(B.cnt.ensure(nB * 4));
    if (s == 0) {
        const uint64_t all = nB + (other ? flat_chunks(other->nbytes) : 0);
        if ((all << FC_SHIFT) >= (1ull << 32)) return fail(h, GENZTOK_E_LIMIT, "chunk too large for the byte-parallel pipeline");
        CU(B.wtok.ensure((all << FC_SHIFT) * 4));
    }
    out->bytes = side.bytes; out->off = side.off; out->n = n;
    out->dsb = B.dsb.as<uint32_t>(); out->st = B.st.as<uint32_t>(); out->tpref = B.tpref.as<uint16_t>(); out->cnt = B.cnt.as<uint32_t>();
    out->wtok = s == 0 ? B.wtok.as<uint32_t>() : d->flat[0].wtok.as<uint32_t>() + (flat_chunks(other->nbytes) << FC_SHIFT);
    out->nB = (uint32_t)nB;
    return GENZTOK_OK;
}

// ---- fixed layout: everything already on the device ------------------------------------------------
int encode_fixed_on_device(genztok_t* h, DeviceCtx* d, cudaStream_t st, const Side& a, const Side* b, int64_t n, int32_t W, uint32_t flags,
                           const genztok_dev_planes_t& P) {
    LaunchScope::cur_stream = st;
    int rc = stream_enter(h, d, st);
    if (rc) return rc;
    const int64_t bytes = a.nbytes + (b ? b->nbytes : 0);
    if (bytes > h->max_chunk_bytes) return fail(h, GENZTOK_E_LIMIT, "chunk of %lld bytes exceeds max_chunk_bytes=%lld", (long long)bytes, (long long)h->max_chunk_bytes);
    rc = ensure_cache(h, d, st, bytes + 32);
    if (rc) return rc;
    if (n <= 0) return GENZTOK_OK;
    CU(d->redo.ensure((size_t)n * 4));
    CU(d->fix.ensure((size_t)n * 4));
    RowArgs A{};
    A.a = a;
    if (b) A.b = *b;
    A.has_pair = b != nullptr;
    A.n_rows = n; A.W = W; A.flags = flags;
    A.ids = P.input_ids; A.mask = P.attention_mask;
    A.tt = (flags & GENZTOK_WANT_TOKEN_TYPE) ? P.token_type_ids : nullptr;
    A.seq = (flags & GENZTOK_WANT_SEQUENCE_ID) ? P.sequence_id : nullptr;
    A.row_len = P.row_len; A.seq_len = P.seq_len; A.status = P.row_status;
    A.redo_list = d->redo.as<uint32_t>(); A.fix_list = d->fix.as<uint32_t>();
    A.eos_i8 = eos_as_i8(d);
    A.pad_i8 = pad_as_i8(d);
    A.D = pick_tile_docs(h, d, a.nbytes, b ? b->nbytes : 0, n, W, true);
    TmaPlanes M;
    // The byte-parallel pipeline (flat.cuh) when the rows are short enough that every word matters; the fused row
    // kernel (which stops reading a document once its row is full) otherwise.
    bool flat = !h->no_flat && !h->no_tma && d->T.specials_distinct && a.nbytes < (1ll << 31) - 65536 && (!b || b->nbytes < (1ll << 31) - 65536) &&
                bytes / n <= 6ll * W;
    if (flat) {
        RowArgs Af = A;
        Af.D = (int32_t)h->flat_rows;
        if (d->over32_pending && cudaEventQuery(d->over32_ev) == cudaSuccess) {
            d->stage32 = d->h_over32[0] * 1000ull <= (unsigned long long)d->over32_rows;      // at most 0.1 % of the rows would take the second pass
            d->over32_pending = false;
        }
        cudaGetLastError();                                           // (cudaErrorNotReady of the query is not an error)
        const int64_t kr_auto = std::max<int64_t>(32, (bytes / n / 3 + 12 + (b ? 4 : 0) + 15) & ~15ll);
        const bool narrow = !h->force_kr && !h->no_stage32 && d->stage32 && kr_auto == 64 && W >= 96;
        if (narrow) h->force_kr = 32;
        flat = setup_tma(h, d, Af, bytes, &M, sizeof(FlatTile));
        if (narrow) h->force_kr = 0;
        if (flat) {
            FlatRowsArgs F{};
            for (int s = 0; s < (b ? 2 : 1); s++) {
                rc = flat_side_setup(h, d, s, s ? *b : a, s ? &a : b, n, s ? &F.b : &F.a);
                if (rc) return rc;
            }
            F.has_pair = b != nullptr; F.n_rows = n; F.W = W; F.D = Af.D; F.ids = A.ids; F.mask = A.mask; F.tt = A.tt;
            F.row_len = A.row_len; F.seq_len = A.seq_len; F.status = A.status; F.redo_list = A.redo_list; F.fix_list = A.fix_list; F.eos_i8 = A.eos_i8; F.pad_i8 = A.pad_i8;
            // cache guard / clear; the document-start bitmaps are zeroed by the same launch
            rc = launch_guard(h, d, st, bytes + 16, 0, F.a.dsb, (uint64_t)F.a.nB * FC_OWN + 2, b ? F.b.dsb : nullptr, b ? (uint64_t)F.b.nB * FC_OWN + 2 : 0);
            if (rc) return rc;
            {
                const unsigned per_side = (unsigned)std::min<int64_t>((n + 256) / 256, (int64_t)d->sm_count * 8);
                LaunchScope ls(h, d, "k_flat_doc_starts");
                CU(launch_pdl(k_flat_doc_starts, dim3(b ? 2 * per_side : per_side), dim3(256), 0, st, d->C, F.a, b ? F.b : F.a, b ? 1 : 0));
            }
            // the pad columns are written by the first k_flat_words launch on the side (tensor stores of [32 x PB] boxes)
            TmaPlanes Mp;
            PadJob J{};
            // (not when the text is tiny next to the planes -- empty documents: a few chunks would have to issue all the boxes)
            if (M.PB > 0 && !h->no_side_pads && (n + 31) / 32 <= 64 * (int64_t)F.a.nB) {
                RowArgs Ap = A;
                Ap.D = 32;
                const int64_t keep_kr = h->force_kr;
                h->force_kr = M.KR;                                   // the same split of the columns as k_flat_rows uses
                const bool okp = setup_tma(h, d, Ap, bytes, &Mp, sizeof(FlatTile)) && Mp.KR == M.KR && Mp.PB == M.PB;
                h->force_kr = keep_kr;
                if (okp) {
                    // rows_pad_pct percent of the pad tiles are left to k_flat_rows (which then needs 32-row tiles too)
                    const int64_t all_tiles = (n + 31) / 32;
                    const int64_t keep = F.D == 32 ? all_tiles * std::min<int64_t>(100, std::max<int64_t>(0, h->rows_pad_pct)) / 100 : 0;
                    J.on = 1; J.n_tiles = (int32_t)(all_tiles - keep); J.W = W; J.D = 32; J.KR = Mp.KR; J.PB = Mp.PB;
                    J.want_tt = (F.has_pair && F.tt) ? 1 : 0; J.pad_id = d->T.pad;
                }
            }
            static const TmaPlanes no_planes{};
            {
                // one launch walks both sides: the resident blocks are split between them in proportion to their chunks
                const bool pads = J.on != 0;                          // every side takes its share of the pad tiles
                FlatWordsArgs WA{};
                auto wk = h->words_minb == 3 ? k_flat_words<3, 1> : (h->words_minb == 2 ? k_flat_words<2, 1> : (h->words_minb == 5 ? k_flat_words<5, 1> : k_flat_words<4, 1>));
                const int64_t wmb = h->words_minb;
                const uint64_t resident = (uint64_t)d->sm_count * (uint64_t)std::max<int64_t>(1, wmb);
                const uint64_t need_a = ((uint64_t)F.a.nB + FW_WARPS - 1) / FW_WARPS, need_b = b ? ((uint64_t)F.b.nB + FW_WARPS - 1) / FW_WARPS : 0;
                uint64_t blocks_a = need_a, blocks_b = need_b;
                if (need_a + need_b > resident) {
                    blocks_a = b ? std::max<uint64_t>(1, resident * need_a / (need_a + need_b)) : resident;
                    blocks_b = b ? std::max<uint64_t>(1, resident - blocks_a) : 0;
                    blocks_a = std::min(blocks_a, need_a); blocks_b = std::min(blocks_b, need_b);
                }
                int64_t alg = 0;
                for (int s = 0; s < (b ? 2 : 1); s++) {
                    const FlatSide& S = s ? F.b : F.a;
                    PadJob Js = J;
                    if (b) {   // pad tiles in proportion to the side's share of the blocks
                        const int32_t first = (int32_t)((int64_t)J.n_tiles * (int64_t)blocks_a / (int64_t)(blocks_a + blocks_b));
                        Js.tile0 = s ? first : 0; Js.n_tiles = s ? J.n_tiles - first : first;
                    }
                    // algorithmic bytes: this side's text, and the pad columns it stores on the side (rows x (W - KR) x (4 + 1 [+ 1]))
                    const int64_t pad_rows = pads ? std::max<int64_t>(0, std::min<int64_t>(n - (int64_t)Js.tile0 * 32, (int64_t)Js.n_tiles * 32)) : 0;
                    alg += (s ? b->nbytes : a.nbytes) + pad_rows * (int64_t)(W - J.KR) * (5 + J.want_tt);
                    Js.l2_policy = (int32_t)h->l2_policy;
                    Js.ratio = (uint32_t)((((uint64_t)std::max<int32_t>(Js.n_tiles, 0) << 20) + S.nB - 1) / S.nB);
                    WA.side[s] = S; WA.job[s] = Js;
                }
                WA.blocks_a = (uint32_t)blocks_a; WA.insert_ok = 1;
                LaunchScope ls(h, d, "k_flat_words", alg);
                const size_t dsm = pads ? tma_const_bytes(J.D, J.PB) : 0;
                if (dsm) CU(cudaFuncSetAttribute(wk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm));
                CU(launch_pdl(wk, dim3((unsigned)(blocks_a + blocks_b)), dim3(FW_THREADS), dsm, st, d->T, d->C, WA, pads ? Mp : no_planes));
                CU(cudaGetLastError());
            }
            // k_flat_rows stores the pad columns of the tiles the side job does not cover (all of them without a side job)
            F.pad_tile0 = J.on ? (uint32_t)J.n_tiles : 0u;
            if (J.on && (int64_t)J.n_tiles >= (n + 31) / 32) M.PB = 0;    // none left: real columns only
            CU(cudaGetLastError());
            rc = launch_bpe(h, d, st);
            if (rc) return rc;
            {
                const bool tt = F.has_pair && F.tt;
                const size_t smem = (M.PB ? tma_const_bytes(F.D, M.PB) : 0) + 8 * r128(sizeof(FlatTile));
                // (the pair instantiation needs its 63 registers: 4 blocks per SM unless asked otherwise)
                const int64_t rmb = h->rows_minb ? h->rows_minb : (F.has_pair ? 3 : 5);
                auto kern = F.has_pair ? (rmb == 3 ? k_flat_rows<3, true> : (rmb == 2 ? k_flat_rows<2, true> : k_flat_rows<4, true>))
                                       : (rmb == 3 ? k_flat_rows<3, false> : (rmb == 2 ? k_flat_rows<2, false> : (rmb == 5 ? k_flat_rows<5, false> : k_flat_rows<4, false>)));
                if (smem > 48 * 1024) CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                int occ = 1;
                CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, smem));
                if (occ < 1) occ = 1;
                const int64_t tiles = (n + F.D - 1) / F.D;
                if (h->rows_grid > 0) occ = std::min<int>(occ, (int)h->rows_grid);
                const int64_t blocks = std::max<int64_t>(1, std::min<int64_t>((tiles + 7) / 8, (int64_t)d->sm_count * occ * h->grid_mult));
                // algorithmic bytes: the document offsets in, the staged columns (and, without the side job, the pad columns) of every plane out
                const int64_t own_pad_rows = M.PB ? std::max<int64_t>(0, n - (int64_t)F.pad_tile0 * 32) : 0;
                LaunchScope ls(h, d, "k_flat_rows", (int64_t)(b ? 2 : 1) * 8 * (n + 1) + (n * (int64_t)M.KR + own_pad_rows * (int64_t)(W - M.KR)) * (5 + (tt ? 1 : 0)));
                CU(launch_pdl(kern, dim3((unsigned)blocks), dim3(256), smem, st, d->T, d->C, F, M));
            }
            CU(cudaGetLastError());
            if (!d->over32_pending && n >= 4096) {                    // sample this call's count of rows longer than 32 tokens
                if (!d->h_over32) CU(cudaHostAlloc(reinterpret_cast<void**>(&d->h_over32), 64, cudaHostAllocDefault));
                if (!d->over32_ev) CU(cudaEventCreateWithFlags(&d->over32_ev, cudaEventDisableTiming));
                CU(cudaMemcpyAsync(d->h_over32, d->C.ctr + C_OVER32, 8, cudaMemcpyDeviceToHost, st));
                CU(cudaEventRecord(d->over32_ev, st));
                d->over32_pending = true; d->over32_rows = n;
            }
        }
    }
    if (!flat) {
        // An empty cache (first call, or after genztok_cache_reset) makes every word new.  The row kernel, a warp per long document,
        // would walk each document until max_len WORDS -- a word not yet through BPE counts as one token -- and every row would be
        // redone afterwards.  Instead the byte-parallel word pass of flat.cuh looks at all the text at once and fills the cache (its
        // word arrays are not used), BPE runs, and the row kernel then finds every word.
        const bool discover = d->cache_empty && !h->no_discovery && a.nbytes < (1ll << 31) - 65536 && (!b || b->nbytes < (1ll << 31) - 65536);
        FlatRowsArgs F{};
        if (discover) {
            for (int s = 0; s < (b ? 2 : 1); s++) {
                rc = flat_side_setup(h, d, s, s ? *b : a, s ? &a : b, n, s ? &F.b : &F.a);
                if (rc) return rc;
            }
            rc = launch_guard(h, d, st, bytes + 16, 0, F.a.dsb, (uint64_t)F.a.nB * FC_OWN + 2, b ? F.b.dsb : nullptr, b ? (uint64_t)F.b.nB * FC_OWN + 2 : 0);
        } else rc = launch_guard(h, d, st, bytes + 16, 0);
        if (rc) return rc;
        if (discover) {
            static const TmaPlanes no_planes{};
            FlatWordsArgs WA{};
            {
                const unsigned per_side = (unsigned)std::min<int64_t>((n + 256) / 256, (int64_t)d->sm_count * 8);
                LaunchScope ls(h, d, "k_flat_doc_starts");
                CU(launch_pdl(k_flat_doc_starts, dim3(b ? 2 * per_side : per_side), dim3(256), 0, st, d->C, F.a, b ? F.b : F.a, b ? 1 : 0));
            }
            WA.side[0] = F.a;
            if (b) WA.side[1] = F.b;
            const uint64_t resident = (uint64_t)d->sm_count * 3;
            const uint64_t need_a = ((uint64_t)F.a.nB + FW_WARPS - 1) / FW_WARPS, need_b = b ? ((uint64_t)F.b.nB + FW_WARPS - 1) / FW_WARPS : 0;
            uint64_t blocks_a = need_a, blocks_b = need_b;
            if (need_a + need_b > resident) {
                blocks_a = b ? std::max<uint64_t>(1, resident * need_a / (need_a + need_b)) : resident;
                blocks_b = b ? std::max<uint64_t>(1, resident - blocks_a) : 0;
                blocks_a = std::min(blocks_a, need_a); blocks_b = std::min(blocks_b, need_b);
            }
            WA.blocks_a = (uint32_t)blocks_a; WA.insert_ok = 1;
            {
                LaunchScope ls(h, d, "k_flat_words_discover", bytes);
                CU(launch_pdl(k_flat_words<3, 1>, dim3((unsigned)(blocks_a + blocks_b)), dim3(FW_THREADS), 0, st, d->T, d->C, WA, no_planes));
            }
            CU(cudaGetLastError());
            rc = launch_bpe(h, d, st);
            if (rc) return rc;
        }
        const bool tma = setup_tma(h, d, A, bytes, &M);
        rc = launch_rows<MODE_FIXED>(h, d, A, st, tma ? "k_rows_fixed_tma" : "k_rows_fixed", n, tma ? &M : nullptr);
        if (rc) return rc;
        rc = launch_bpe(h, d, st);
        if (rc) return rc;
    }
    RowArgs R = A;
    R.row_list = d->redo.as<uint32_t>();
    rc = launch_rows<MODE_FIXED>(h, d, R, st, "k_rows_fixed_redo", std::min<int64_t>(n, (int64_t)d->sm_count * 64));
    if (rc) return rc;
    if (b && (A.tt || A.seq || A.status || A.seq_len)) {
        PostArgs Q{};
        Q.ids = P.input_ids; Q.W = W; Q.n_rows = n; Q.row_list = d->fix.as<uint32_t>();
        Q.has_pair = 1; Q.tt = A.tt; Q.seq = A.seq; Q.seq_len = P.seq_len; Q.status = P.row_status;
        Q.has_max_len = 1; Q.max_len = W; Q.padding = 1; Q.truncation = 1; Q.eos_i8 = A.eos_i8; Q.pad_i8 = A.pad_i8;
        LaunchScope ls(h, d, "k_post_rows_fix");
        k_post_rows<<<d->sm_count, 256, 0, st>>>(d->T, Q, d->C.ctr + C_FIX);
        CU(cudaGetLastError());
    }
    d->cache_empty = false;
    return stream_leave(h, d, st);
}

// ---- long documents as windows (window.cuh) -------------------------------------------------------------
// Token stream of one side: [bos] T [eos] of every document, untruncated, ragged at off[m+1] (the ragged pipeline with max_len
// None, without the mask and k_post_rows).  Reads the stream's size back to size `ids` (synchronises).  offs: also the tokens'
// byte offsets, aligned with ids ((0, 0) for the framing).
int token_stream(genztok_t* h, DeviceCtx* d, cudaStream_t st, const Side& s, int64_t m, DevBuf& ids, DevBuf& off, DevBuf* offs) {
    CU(d->redo.ensure((size_t)m * 4)); CU(d->fix.ensure((size_t)m * 4));
    CU(d->L.ensure((size_t)m * 4)); CU(d->keep.ensure((size_t)m * 4)); CU(d->out_len.ensure((size_t)m * 8)); CU(d->tail.ensure((size_t)m));
    CU(off.ensure((size_t)(m + 1) * 8));
    { LaunchScope ls(h, d, "k_reset_lists"); k_reset_lists<<<1, 1, 0, st>>>(d->C); }
    RowArgs A{};
    A.a = s; A.n_rows = m; A.L = d->L.as<int32_t>(); A.redo_list = d->redo.as<uint32_t>(); A.fix_list = d->fix.as<uint32_t>();
    A.eos_i8 = eos_as_i8(d); A.pad_i8 = pad_as_i8(d);
    A.D = pick_tile_docs(h, d, s.nbytes, 0, m, 0, false);
    int rc = launch_rows<MODE_COUNT>(h, d, A, st, "k_rows_count", m);
    if (rc) return rc;
    rc = launch_bpe(h, d, st);
    if (rc) return rc;
    RowArgs R = A;
    R.row_list = d->redo.as<uint32_t>();
    rc = launch_rows<MODE_COUNT>(h, d, R, st, "k_rows_count_redo", std::min<int64_t>(m, (int64_t)d->sm_count * 64));
    if (rc) return rc;
    LenArgs LA{d->L.as<int32_t>(), m, 0, 0, 0, 0, d->keep.as<int32_t>(), d->out_len.as<int64_t>(), d->tail.as<uint8_t>(), nullptr, nullptr, nullptr};
    { LaunchScope ls(h, d, "k_row_lens"); k_row_lens<<<(unsigned)std::min<int64_t>((m + 255) / 256, 4096), 256, 0, st>>>(LA); }
    rc = launch_scan(h, d, st, d->out_len.as<int64_t>(), off.as<int64_t>(), m);
    if (rc) return rc;
    int64_t total = 0;
    CU(cudaMemcpyAsync(&total, off.as<int64_t>() + m, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(ids.ensure((size_t)total * 4 + 16));
    { LaunchScope ls(h, d, "k_reset_lists"); k_reset_lists<<<1, 1, 0, st>>>(d->C); }
    RowArgs E = A;
    E.ids = ids.as<int32_t>(); E.row_off = off.as<int64_t>(); E.keep = d->keep.as<int32_t>();
    if (offs) {
        CU(offs->ensure((size_t)total * 8 + 16));
        CU(cudaMemsetAsync(offs->p, 0, (size_t)total * 8, st));
        E.offs = offs->as<int32_t>(); E.plen = d->len_arena.as<uint16_t>();
    }
    return launch_rows<MODE_RAGGED>(h, d, E, st, offs ? "k_rows_ragged_offsets" : "k_rows_ragged", m);
}

WinArgs window_args(DeviceCtx* d, bool pair, int64_t n, int32_t W, int32_t s) {
    WinArgs A{};
    A.ids_a = d->win.ids[0].as<int32_t>(); A.off_a = d->win.off[0].as<int64_t>();
    if (pair) { A.ids_b = d->win.ids[1].as<int32_t>(); A.off_b = d->win.off[1].as<int64_t>(); }
    A.offs_a = d->win.offs[0].as<int2>(); A.offs_b = pair ? d->win.offs[1].as<int2>() : nullptr;
    A.len_a = d->win.len[0].as<int32_t>(); A.len_b = pair ? d->win.len[1].as<int32_t>() : nullptr;
    A.n_docs = n; A.W = W; A.stride = s;
    A.ctr = d->C.ctr;
    A.eos_i8 = eos_as_i8(d); A.pad_i8 = pad_as_i8(d);
    return A;
}

// Step 1: both token streams, the windows of every document, d_win_off[n+1] and their total (synchronises).  The caller has
// sized the word cache for the chunk (ensure_cache) and n >= 1.  offs: the streams carry token offsets too (offset_mapping).
// strategy (a pair truncation strategy, PAIR_*): the streams only; one row per document, *n_win = n, d_win_off is not used.
int windows_layout(genztok_t* h, DeviceCtx* d, cudaStream_t st, const Side& a, const Side* b, int64_t n, int32_t W, int32_t s, int32_t strategy,
                   bool offs, int64_t* d_win_off, int64_t* n_win) {
    d->win.n_win = -1;                                               // the streams are about to change
    int rc = offs ? ensure_piece_lens(h, d, st) : GENZTOK_OK;
    if (rc) return rc;
    rc = launch_guard(h, d, st, a.nbytes + (b ? b->nbytes : 0) + 16, 0);
    if (rc) return rc;
    rc = token_stream(h, d, st, a, n, d->win.ids[0], d->win.off[0], offs ? &d->win.offs[0] : nullptr);
    if (!rc && b) rc = token_stream(h, d, st, *b, n, d->win.ids[1], d->win.off[1], offs ? &d->win.offs[1] : nullptr);
    if (rc) return rc;
    d->cache_empty = false;
    if (strategy) { *n_win = n; return GENZTOK_OK; }
    CU(d->win.count.ensure((size_t)n * 8));
    WinArgs A = window_args(d, b != nullptr, n, W, s);
    A.count = d->win.count.as<int64_t>();
    { LaunchScope ls(h, d, "k_window_count"); k_window_count<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)d->sm_count * 8), 256, 0, st>>>(A); }
    CU(cudaGetLastError());
    rc = launch_scan(h, d, st, d->win.count.as<int64_t>(), d_win_off, n);
    if (rc) return rc;
    CU(cudaMemcpyAsync(n_win, d_win_off + n, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return GENZTOK_OK;
}

// Step 2: the K windows' planes and maps from the streams step 1 left (does not synchronise).  win_doc = doc_base + document.
// With GENZTOK_WANT_OFFSETS in flags, P.offsets receives [K, W, 2] token offsets (step 1 must have run with offsets).
// strategy: the K = n rows of a pair truncation strategy (k_pair_rows), or with STREAMS_CAPPED the K = n reference rows of the capped
// streams dropout_layout left (k_dropout_rows); d_win_off, win_doc and win_start are not used.
int windows_write(genztok_t* h, DeviceCtx* d, cudaStream_t st, bool pair, int64_t n, int32_t W, int32_t s, int32_t strategy, uint32_t flags,
                  const int64_t* d_win_off, int64_t K, const genztok_dev_planes_t& P, int64_t* win_doc, int32_t* win_start, int64_t doc_base) {
    if (K <= 0) return GENZTOK_OK;
    if (K >= (1ll << 32)) return fail(h, GENZTOK_E_LIMIT, "%lld windows in one chunk", (long long)K);
    CU(d->win.fix.ensure((size_t)K * 4));
    { LaunchScope ls(h, d, "k_reset_lists"); k_reset_lists<<<1, 1, 0, st>>>(d->C); }
    WinArgs A = window_args(d, pair, n, W, s);
    A.win_off = d_win_off; A.n_win = K; A.doc_base = doc_base; A.strategy = strategy;
    A.ids = P.input_ids; A.mask = P.attention_mask; A.row_len = P.row_len;
    if (pair) {
        A.tt = (flags & GENZTOK_WANT_TOKEN_TYPE) ? P.token_type_ids : nullptr;
        A.seq = (flags & GENZTOK_WANT_SEQUENCE_ID) ? P.sequence_id : nullptr;
        A.seq_len = P.seq_len; A.status = P.row_status;
    }
    A.win_doc = win_doc; A.win_start = win_start; A.fix_list = d->win.fix.as<uint32_t>();
    const bool offs = (flags & GENZTOK_WANT_OFFSETS) != 0;            // (P.offsets is read only then: older callers' structs end before it)
    if (offs) A.offs = P.offsets;
    auto aligned = [](const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; };
    const bool quad = (W & 3) == 0 && aligned(A.ids, 16) && aligned(A.mask, 4) && aligned(A.tt, 4) && aligned(A.seq, 4) && aligned(A.offs, 16);
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((K + 7) / 8, (int64_t)d->sm_count * 8));
    {
        // algorithmic bytes: the planes and per-window values written (the windows' tokens are read from the streams, mostly in L2)
        const int64_t alg = K * (int64_t)W * (5 + (A.tt ? 1 : 0) + (A.seq ? 1 : 0) + (offs ? 8 : 0)) + K * (4 + 8 + 4 + (pair ? 5 : 0));
        LaunchScope ls(h, d, strategy == STREAMS_CAPPED ? "k_dropout_rows" : strategy ? (offs ? "k_pair_rows_offsets" : "k_pair_rows")
                                                                                : offs ? "k_window_rows_offsets" : "k_window_rows", alg);
        if (strategy == STREAMS_CAPPED) {
            if (pair) { if (quad) k_dropout_rows<true, true><<<grid, 256, 0, st>>>(d->T, A); else k_dropout_rows<false, true><<<grid, 256, 0, st>>>(d->T, A); }
            else { if (quad) k_dropout_rows<true, false><<<grid, 256, 0, st>>>(d->T, A); else k_dropout_rows<false, false><<<grid, 256, 0, st>>>(d->T, A); }
        } else if (strategy) {
            if (offs) { if (quad) k_window_rows<true, true, true, true><<<grid, 256, 0, st>>>(d->T, A); else k_window_rows<false, true, true, true><<<grid, 256, 0, st>>>(d->T, A); }
            else { if (quad) k_window_rows<true, true, false, true><<<grid, 256, 0, st>>>(d->T, A); else k_window_rows<false, true, false, true><<<grid, 256, 0, st>>>(d->T, A); }
        } else if (offs) {
            if (pair) { if (quad) k_window_rows<true, true, true><<<grid, 256, 0, st>>>(d->T, A); else k_window_rows<false, true, true><<<grid, 256, 0, st>>>(d->T, A); }
            else { if (quad) k_window_rows<true, false, true><<<grid, 256, 0, st>>>(d->T, A); else k_window_rows<false, false, true><<<grid, 256, 0, st>>>(d->T, A); }
        } else {
            if (pair) { if (quad) k_window_rows<true, true><<<grid, 256, 0, st>>>(d->T, A); else k_window_rows<false, true><<<grid, 256, 0, st>>>(d->T, A); }
            else { if (quad) k_window_rows<true, false><<<grid, 256, 0, st>>>(d->T, A); else k_window_rows<false, false><<<grid, 256, 0, st>>>(d->T, A); }
        }
    }
    CU(cudaGetLastError());
    if (pair && (A.tt || A.seq || A.seq_len || A.status)) {
        PostArgs Q{};
        Q.ids = P.input_ids; Q.W = W; Q.n_rows = K; Q.row_list = A.fix_list;
        Q.has_pair = 1; Q.tt = A.tt; Q.seq = A.seq; Q.seq_len = A.seq_len; Q.status = A.status;
        Q.has_max_len = 1; Q.max_len = W; Q.padding = 1; Q.truncation = 1; Q.eos_i8 = A.eos_i8; Q.pad_i8 = A.pad_i8;
        const bool keep2 = strategy && strategy != STREAMS_CAPPED;    // (status 2 exists only for the strategies)
        LaunchScope ls(h, d, strategy == STREAMS_CAPPED ? "k_post_rows_dropout" : strategy ? "k_post_rows_pairs" : "k_post_rows_windows");
        if (keep2) k_post_rows<true><<<d->sm_count, 256, 0, st>>>(d->T, Q, d->C.ctr + C_FIX);
        else k_post_rows<<<d->sm_count, 256, 0, st>>>(d->T, Q, d->C.ctr + C_FIX);
        CU(cudaGetLastError());
    }
    return GENZTOK_OK;
}

// BPE-dropout, step 1: the two capped token streams of n documents (k_dropout_stream) into d->win.ids / d->win.len, for
// windows_write(..., STREAMS_CAPPED, ...).  Row d's key is d_keys[d] (device memory), or key_base + d.  Does not synchronise; the
// buffers grow (cudaMalloc) only when a call is larger than every earlier one on the device.  The word cache is not used.
int dropout_layout(genztok_t* h, DeviceCtx* d, cudaStream_t st, const Side& a, const Side* b, int64_t n, int32_t W, double p, uint64_t seed,
                   const int64_t* d_keys, int64_t key_base) {
    d->win.n_win = -1;                                               // the window streams are about to change
    const size_t slots = (size_t)n * (size_t)(W + 2);
    const int64_t nbytes = a.nbytes + (b ? b->nbytes : 0);
    for (int s = 0; s < (b ? 2 : 1); s++) { CU(d->win.ids[s].ensure(slots * 4 + 16)); CU(d->win.len[s].ensure((size_t)n * 4 + 16)); }
    CU(d->win.drop_scratch.ensure((size_t)nbytes * 8 + 64));
    DropArgs A{};
    A.a = a; if (b) A.b = *b;
    A.n = n; A.cap = W;
    A.s0 = mix64(seed ^ DROP_K); A.thr = (uint64_t)std::floor(p * 4294967296.0);
    A.row_keys = d_keys; A.key_base = key_base;
    A.ids_a = d->win.ids[0].as<int32_t>(); A.len_a = d->win.len[0].as<int32_t>();
    if (b) { A.ids_b = d->win.ids[1].as<int32_t>(); A.len_b = d->win.len[1].as<int32_t>(); }
    A.scratch = d->win.drop_scratch.as<uint32_t>(); A.b_base = a.nbytes; A.nbytes = nbytes;
    A.ctr = d->C.ctr;
    const int64_t warps = b ? 2 * n : n;
    {
        LaunchScope ls(h, d, "k_dropout_stream", nbytes + (int64_t)slots * 4 * (b ? 2 : 1));
        k_dropout_stream<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((warps + 7) / 8, (int64_t)d->sm_count * 64)), 256, 0, st>>>(d->T, A);
    }
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

void* host_pool_get(genztok_t* h, size_t bytes, size_t* got = nullptr) {
    if (bytes == 0) bytes = 16;
    {
        std::lock_guard<std::mutex> l(h->pool_mu);
        auto it = h->host_pool.lower_bound(bytes);
        if (it != h->host_pool.end() && it->first <= bytes + bytes / 4 + 4096) {
            void* p = it->second;
            if (got) *got = it->first;
            h->host_pool_bytes -= it->first;
            h->host_pool.erase(it);
            return p;
        }
    }
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (got) *got = bytes;
    return p;
}
void host_pool_put(genztok_t* h, void* p, size_t bytes) {
    std::lock_guard<std::mutex> l(h->pool_mu);
    if (h->host_pool_bytes + bytes > (size_t)8 << 30) { h->plane_meta.erase(p); cudaFreeHost(p); return; }
    h->host_pool.insert({bytes, p});
    h->host_pool_bytes += bytes;
}

// A growable array in pinned host memory (from the handle's pool): what a device worker collects ragged results in.  Device to
// host copies into pageable memory are staged by the driver at a fraction of the link's rate; resize() does not initialise.
template <class T>
struct PinnedVec {
    genztok_t* h = nullptr; T* p = nullptr; size_t n = 0, cap_bytes = 0;
    PinnedVec() = default;
    PinnedVec(const PinnedVec&) = delete;
    PinnedVec& operator=(const PinnedVec&) = delete;
    ~PinnedVec() { if (p) host_pool_put(h, p, cap_bytes); }
    bool resize(size_t m) {
        if (m * sizeof(T) > cap_bytes) {
            size_t got = 0;
            const size_t want = std::max<size_t>(m * sizeof(T) + m * sizeof(T) / 2, 1 << 16);
            T* q = reinterpret_cast<T*>(host_pool_get(h, (want + 4095) & ~(size_t)4095, &got));
            if (!q) return false;
            { std::lock_guard<std::mutex> l(h->pool_mu); h->plane_meta.erase(q); }   // (it is about to hold other data than a padded plane)
            if (n) memcpy(q, p, n * sizeof(T));
            if (p) host_pool_put(h, p, cap_bytes);
            p = q; cap_bytes = got;
        }
        n = m;
        return true;
    }
    bool reserve(size_t m) { const size_t keep = n; if (m * sizeof(T) > cap_bytes) { if (!resize(m)) return false; n = keep; } return true; }
    T* data() { return p; }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
};

struct OutBlock {
    std::vector<std::pair<void*, size_t>> pinned;   // returned to the pool on free
    std::vector<void*> mallocs;
};

template <class T>
T* out_alloc(genztok_t* h, OutBlock* ob, size_t count) {
    size_t bytes = std::max<size_t>(count * sizeof(T), 16);
    bytes = (bytes + 4095) & ~(size_t)4095;
    void* p = host_pool_get(h, bytes);
    if (!p) return nullptr;
    ob->pinned.push_back({p, bytes});
    return reinterpret_cast<T*>(p);
}

// Gives a result block's buffers back (the pinned ones to the pool) and deletes it.
void release_block(genztok_t* h, OutBlock* ob) {
    for (auto& pr : ob->pinned) host_pool_put(h, pr.first, pr.second);
    for (void* p : ob->mallocs) free(p);
    delete ob;
}

// The same for the result of a call that failed: what its pooled planes hold is unknown, so their plane_meta records go too.  (A
// result that its owner frees keeps them: a recycled fixed-layout plane copies only the columns its record says can differ.)
void discard_block(genztok_t* h, OutBlock* ob) {
    for (auto& pr : ob->pinned) h->plane_meta.erase(pr.first);
    release_block(h, ob);
}

// genztok_free_encoded / genztok_free_text
template <class Out>
void free_result(genztok_t* h, Out* out) {
    if (!out || !out->_owner) return;
    { std::lock_guard<std::mutex> lk(h->mu); release_block(h, reinterpret_cast<OutBlock*>(out->_owner)); }
    memset(out, 0, sizeof *out);
}

}  // namespace

// ================================================================================================
extern "C" {

const char* genztok_version(void) { return "genztok-b200 0.6 (sm_100a)"; }

const char* genztok_last_error(const genztok_t* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int genztok_create(const char* vocab_path, const char* bpe_path, const char* const specials_utf8[5], const int* device_ids, int n_devices,
                   genztok_t** out) {
    if (!vocab_path || !bpe_path || !out || n_devices < 0) return fail(nullptr, GENZTOK_E_INVALID, "genztok_create: bad arguments");
    genztok_t* h = new genztok();
    if (!h->H.build(vocab_path, bpe_path, specials_utf8)) {
        g_create_err = h->H.err;
        int code = h->H.err_code;
        delete h;
        return code;
    }
    for (int i = 0; i < n_devices; i++) {
        DeviceCtx* d = new DeviceCtx();
        d->device = device_ids ? device_ids[i] : i;
        h->devs.push_back(d);
        int rc = init_device(h, d);
        if (rc) {
            g_create_err = h->err;
            genztok_destroy(h);
            return rc;
        }
    }
    *out = h;
    return GENZTOK_OK;
}

void genztok_destroy(genztok_t* h) {
    if (!h) return;
    for (DeviceCtx* d : h->devs) {
        cudaSetDevice(d->device);
        if (d->stream) cudaStreamSynchronize(d->stream);
        for (void* p : d->table_allocs) cudaFree(p);
        for (DevBuf* b : {&d->text, &d->toff, &d->pair, &d->poff, &d->ids, &d->mask, &d->tt, &d->seq, &d->row_len, &d->seq_len, &d->tt_len,
                          &d->status, &d->L, &d->keep, &d->out_len, &d->row_off, &d->tail, &d->redo, &d->fix, &d->misc, &d->nwA, &d->nwB, &d->span_cnt, &d->span_off, &d->spans, &d->scan_tmp, &d->prep_out, &d->dec_lead, &d->tok_flag, &d->tok_len, &d->tok_pos, &d->slots,
                          &d->key_arena, &d->tok_arena, &d->pending, &d->ctr, &d->rank_scratch, &d->dec_stat})
            b->release();
        for (auto& e : d->events) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
        for (auto e : d->free_events) cudaEventDestroy(e);
        for (auto& sg : d->stage) {
            for (DevBuf* b : {&sg.text, &sg.toff, &sg.pair, &sg.poff, &sg.ids, &sg.mask, &sg.tt, &sg.seq, &sg.row_len, &sg.seq_len, &sg.status, &sg.extent}) b->release();
            for (cudaEvent_t e : {sg.h2d, sg.k, sg.d2h}) if (e) cudaEventDestroy(e);
        }
        if (d->s_in) cudaStreamDestroy(d->s_in);
        if (d->s_out) cudaStreamDestroy(d->s_out);
        if (d->h_extent) cudaFreeHost(d->h_extent);
        if (d->h_over32) cudaFreeHost(d->h_over32);
        if (d->over32_ev) cudaEventDestroy(d->over32_ev);
        if (d->last_done) cudaEventDestroy(d->last_done);
        d->synth_len.release();
        for (DevBuf* b : {&d->win.ids[0], &d->win.ids[1], &d->win.off[0], &d->win.off[1], &d->win.count, &d->win.woff, &d->win.fix, &d->win.doc, &d->win.start,
                          &d->win.offs[0], &d->win.offs[1], &d->win.plane_offs, &d->win.len[0], &d->win.len[1], &d->win.drop_scratch, &d->win.drop_keys})
            b->release();
        for (auto& fb : d->flat) for (DevBuf* b : {&fb.dsb, &fb.st, &fb.tpref, &fb.cnt, &fb.wtok}) b->release();
        if (d->stream) cudaStreamDestroy(d->stream);
        delete d;
    }
    for (auto& kv : h->host_pool) cudaFreeHost(kv.second);
    delete h;
}

int64_t genztok_vocab_size(const genztok_t* h) { return (int64_t)h->H.enc_keys.size(); }
int genztok_special_ids(const genztok_t* h, int32_t out[5]) {
    for (int i = 0; i < 5; i++) out[i] = h->H.special_id[i];
    return GENZTOK_OK;
}
int64_t genztok_encoder_count(const genztok_t* h) { return (int64_t)h->H.enc_keys.size(); }
int genztok_encoder_entry(const genztok_t* h, int64_t i, const uint8_t** key, int64_t* key_len, int32_t* id) {
    if (i < 0 || i >= (int64_t)h->H.enc_keys.size()) return GENZTOK_E_INVALID;
    *key = (const uint8_t*)h->H.enc_keys[(size_t)i].data();
    *key_len = (int64_t)h->H.enc_keys[(size_t)i].size();
    *id = h->H.enc_vals[(size_t)i];
    return GENZTOK_OK;
}
int32_t genztok_encoder_get(const genztok_t* h, const uint8_t* key, int64_t key_len) {
    return h->H.enc_get(std::string((const char*)key, (size_t)key_len), -1);
}
int genztok_decoder_get(const genztok_t* h, int64_t id, const uint8_t** key, int64_t* key_len) {
    *key = nullptr; *key_len = 0;
    if (id < 0 || id >= h->H.n_ids || h->H.decoder[(size_t)id] < 0) return GENZTOK_OK;
    const std::string& s = h->H.enc_keys[(size_t)h->H.decoder[(size_t)id]];
    *key = (const uint8_t*)s.data(); *key_len = (int64_t)s.size();
    return GENZTOK_OK;
}
int64_t genztok_merge_count(const genztok_t* h) { return (int64_t)h->H.merge_lines.size(); }
int genztok_merge_line(const genztok_t* h, int64_t i, const uint8_t** line, int64_t* line_len) {
    if (i < 0 || i >= (int64_t)h->H.merge_lines.size()) return GENZTOK_E_INVALID;
    *line = (const uint8_t*)h->H.merge_lines[(size_t)i].data();
    *line_len = (int64_t)h->H.merge_lines[(size_t)i].size();
    return GENZTOK_OK;
}
int32_t genztok_rank_get(const genztok_t* h, const uint8_t* l, int64_t l_len, const uint8_t* r, int64_t r_len) {
    return h->H.rank_get(std::string((const char*)l, (size_t)l_len), std::string((const char*)r, (size_t)r_len));
}

int genztok_device_count(const genztok_t* h) { return (int)h->devs.size(); }
int64_t genztok_launch_count(const genztok_t* h) { return h->launches.load(); }

void* genztok_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void genztok_host_free(void* p) { if (p) cudaFreeHost(p); }

int genztok_set_option(genztok_t* h, const char* name, int64_t value) {
    std::string n = name ? name : "";
    if (n == "fixed_cache") {
        h->fixed_cache = value;
    } else if (n == "max_chunk_bytes") {
        for (DeviceCtx* d : h->devs) if (d->cache_ready) return fail(h, GENZTOK_E_INVALID, "max_chunk_bytes must be set before the first encode");
        if (value < 4096 || value > (1ll << 29)) return fail(h, GENZTOK_E_INVALID, "max_chunk_bytes must be in [4 KiB, 512 MiB]");
        h->max_chunk_bytes = value;
    } else if (n == "chunk_rows") {
        if (value < 1) return fail(h, GENZTOK_E_INVALID, "chunk_rows < 1");
        h->chunk_rows = value;
    } else if (n == "group") {
        if (value < 0 || value > 32) return fail(h, GENZTOK_E_INVALID, "group (documents per warp tile) must be 0 (auto) or 1..32");
        h->force_group = value;
    } else if (n == "grid_mult") {
        if (value < 1 || value > 1024) return fail(h, GENZTOK_E_INVALID, "grid_mult must be in 1..1024");
        h->grid_mult = value;
    } else if (n == "wide_rows") {
        h->force_wide = value;
        for (DeviceCtx* d : h->devs) d->force_wide = value != 0;
    } else if (n == "no_flat") {
        h->no_flat = value;
    } else if (n == "no_stage32") {
        h->no_stage32 = value;
    } else if (n == "no_discovery") {
        h->no_discovery = value;
    } else if (n == "flat_rows") {
        if (value < 1 || value > 32) return fail(h, GENZTOK_E_INVALID, "flat_rows must be in 1..32");
        h->flat_rows = value;
    } else if (n == "no_side_pads") {
        h->no_side_pads = value;
    } else if (n == "pad_box_cols") {
        if (value < 0 || value > 256 || (value & 15)) return fail(h, GENZTOK_E_INVALID, "pad_box_cols must be 0 or a multiple of 16 up to 256");
        h->pad_box_cols = value;
    } else if (n == "decode_write") {
        h->decode_write = value;
    } else if (n == "decode_wide_max") {
        h->decode_wide_max = value;
    } else if (n == "no_copy_kernel") {
        h->no_copy_kernel = value;
    } else if (n == "copy_round") {
        if (value != 32 && value != 64) return fail(h, GENZTOK_E_INVALID, "copy_round must be 32 or 64");
        h->copy_round = value;
    } else if (n == "copy_blocks") {
        if (value < 1 || value > 4096) return fail(h, GENZTOK_E_INVALID, "copy_blocks must be in 1..4096");
        h->copy_blocks = value;
    } else if (n == "l2_policy") {
        h->l2_policy = value;
    } else if (n == "rows_pad_pct") {
        if (value < 0 || value > 100) return fail(h, GENZTOK_E_INVALID, "rows_pad_pct must be in 0..100");
        h->rows_pad_pct = value;
    } else if (n == "rows_grid") {
        h->rows_grid = value;
    } else if (n == "rows_minb") {
        h->rows_minb = value;
    } else if (n == "words_minb") {
        h->words_minb = value;
    } else if (n == "no_tma") {
        h->no_tma = value;
    } else if (n == "no_fixed_decode") {
        h->no_fixed_decode = value;
    } else if (n == "no_token_decode") {
        h->no_token_decode = value;
    } else if (n == "tma_columns") {
        if (value < 0 || value > 256 || (value & 15)) return fail(h, GENZTOK_E_INVALID, "tma_columns must be 0 (auto) or a multiple of 16 up to 256");
        h->force_kr = value;
    } else return fail(h, GENZTOK_E_INVALID, "unknown option %s", n.c_str());
    return GENZTOK_OK;
}

int genztok_cache_reset(genztok_t* h) {
    std::lock_guard<std::mutex> lk(h->mu);
    for (DeviceCtx* d : h->devs) {
        if (!d->cache_ready) continue;
        CU(cudaSetDevice(d->device));
        LaunchScope::cur_stream = d->stream;
        int rc = launch_guard(h, d, d->stream, 0, 1);
        if (rc) return rc;
        CU(cudaStreamSynchronize(d->stream));
        d->cache_empty = true;
    }
    return GENZTOK_OK;
}

int genztok_set_profiling(genztok_t* h, int on) {
    for (DeviceCtx* d : h->devs) d->profiling = on != 0;
    return GENZTOK_OK;
}

int64_t genztok_profile_report(genztok_t* h, char* buf, int64_t cap, int reset) {
    std::lock_guard<std::mutex> lk(h->mu);
    for (DeviceCtx* d : h->devs) {
        cudaSetDevice(d->device);
        cudaDeviceSynchronize();
        for (auto& e : d->events) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) {
                auto& acc = h->prof_acc[h->prof_names[(size_t)e.name]];
                acc.launches += 1; acc.ms += ms; acc.alg += e.alg;
            } else cudaGetLastError();
            d->free_events.push_back(e.a); d->free_events.push_back(e.b);
        }
        d->events.clear();
    }
    std::string s = "{";
    bool first = true;
    for (auto& kv : h->prof_acc) {
        char t[256];
        snprintf(t, sizeof t, "%s\"%s\": {\"launches\": %lld, \"ms\": %.6f, \"alg_bytes\": %lld}", first ? "" : ", ", kv.first.c_str(), (long long)kv.second.launches,
                 kv.second.ms, (long long)kv.second.alg);
        s += t; first = false;
    }
    s += "}";
    if (reset) h->prof_acc.clear();
    if (buf && cap > 0) { size_t n = std::min<size_t>(s.size(), (size_t)cap - 1); memcpy(buf, s.data(), n); buf[n] = 0; }
    return (int64_t)s.size() + 1;
}

// ---- encode -----------------------------------------------------------------------------------------
}  // extern "C"

namespace {

// The truncation strategy of flags (PAIR_*, or 0 for the reference cut) into *strategy, after the checks both encode forms share:
// at most one strategy bit, and the fixed layout (max_len >= 4; the host form also padding and truncation, and no spans).
int pair_strategy(genztok_t* h, uint32_t flags, int32_t max_len, bool fixed, int32_t* strategy) {
    const uint32_t bits = flags & (GENZTOK_LONGEST_FIRST | GENZTOK_ONLY_FIRST | GENZTOK_ONLY_SECOND);
    *strategy = bits == GENZTOK_LONGEST_FIRST ? PAIR_LONGEST_FIRST : bits == GENZTOK_ONLY_FIRST ? PAIR_ONLY_FIRST : bits == GENZTOK_ONLY_SECOND ? PAIR_ONLY_SECOND : 0;
    if (!bits) return GENZTOK_OK;
    if (!*strategy) return fail(h, GENZTOK_E_INVALID, "at most one truncation strategy (GENZTOK_LONGEST_FIRST, GENZTOK_ONLY_FIRST, GENZTOK_ONLY_SECOND)");
    if (max_len < 4) return fail(h, GENZTOK_E_INVALID, "a truncation strategy needs max_len >= 4 (got %s)", max_len == GENZTOK_MAX_LEN_NONE ? "None" : std::to_string(max_len).c_str());
    if (!fixed) return fail(h, GENZTOK_E_INVALID, "a truncation strategy needs the fixed layout: padding and truncation, without return_offset spans");
    return GENZTOK_OK;
}

}  // namespace

extern "C" {

int genztok_encode_device(genztok_t* h, int dev, const uint8_t* d_text, const int64_t* d_text_off, int64_t text_bytes, const uint8_t* d_pair,
                          const int64_t* d_pair_off, int64_t pair_bytes, int64_t n, int32_t max_len, uint32_t flags,
                          const genztok_dev_planes_t* planes, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    int32_t strategy = 0;
    int rc = pair_strategy(h, flags, max_len, true, &strategy);
    if (rc) return rc;
    if (strategy && (flags & (GENZTOK_WANT_OFFSETS | GENZTOK_WANT_SPANS)))
        return fail(h, GENZTOK_E_INVALID, "genztok_encode_device: offsets and spans are not available with a truncation strategy");
    if (strategy && (!planes || !planes->input_ids || !planes->attention_mask || !planes->row_len))
        return fail(h, GENZTOK_E_INVALID, "genztok_encode_device: a truncation strategy needs input_ids, attention_mask and row_len");
    if (flags & GENZTOK_WANT_OFFSETS) return fail(h, GENZTOK_E_INVALID, "offsets are not available in the fixed device layout; use genztok_encode_windows_device");
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d (handle has %d)", dev, (int)h->devs.size());
    if (!planes || !planes->input_ids || n < 0 || !d_text_off || (text_bytes > 0 && !d_text)) return fail(h, GENZTOK_E_INVALID, "genztok_encode_device: bad arguments");
    if (max_len < 1) return fail(h, GENZTOK_E_INVALID, "genztok_encode_device needs max_len >= 1 (fixed layout)");
    if (((uintptr_t)d_text & 15) || ((uintptr_t)d_pair & 15)) return fail(h, GENZTOK_E_INVALID, "device text buffers must be 16-byte aligned");
    if (flags & GENZTOK_WANT_SPANS) return fail(h, GENZTOK_E_INVALID, "spans are not available in the fixed device layout");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    Side a{d_text, d_text_off, text_bytes}, b{d_pair, d_pair_off, pair_bytes};
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    if (strategy && d_pair_off) {
        // the rows of a truncation strategy: both token streams (sized by a read-back: synchronises), then one k_pair_rows launch
        LaunchScope::cur_stream = st;
        const int64_t bytes = text_bytes + pair_bytes;
        if (bytes > h->max_chunk_bytes) return fail(h, GENZTOK_E_LIMIT, "chunk of %lld bytes exceeds max_chunk_bytes=%lld", (long long)bytes, (long long)h->max_chunk_bytes);
        rc = stream_enter(h, d, st);
        if (rc) return rc;
        if (n > 0) {
            int64_t K = 0;
            rc = ensure_cache(h, d, st, bytes + 32);
            if (!rc) rc = windows_layout(h, d, st, a, &b, n, max_len, 0, strategy, false, nullptr, &K);
            if (!rc) rc = windows_write(h, d, st, true, n, max_len, 0, strategy, flags, nullptr, K, *planes, nullptr, nullptr, 0);
            if (rc) return rc;
        }
        return stream_leave(h, d, st);
    }
    if (!fixed_fits(d, max_len)) return fail(h, GENZTOK_E_LIMIT, "max_len=%d does not fit the fixed-layout kernel; use genztok_encode", max_len);
    return encode_fixed_on_device(h, d, st, a, d_pair_off ? &b : nullptr, n, max_len, flags, *planes);
}

void genztok_free_encoded(genztok_t* h, genztok_encoded_t* out) { free_result(h, out); }

}  // extern "C"

namespace {

// Everything one device does for its contiguous range of rows [rb, re): chunk loop, H2D, kernels, D2H.
// Fixed layout: results land in the caller-visible pinned planes of `out` at the rows' final places.
// Ragged layout: flat planes are collected in `part` (offsets relative to the part) and stitched by the caller.
struct EncodeJob {
    const uint8_t* text; const int64_t* text_off; const uint8_t* pair; const int64_t* pair_off;
    int32_t max_len; int padding, truncation; uint32_t flags;
    bool has_pair, has_max_len, want_spans, fixed, want_tt, want_seq;
    bool want_offs;                // offset_mapping: the ragged pipeline writes token offsets beside the ids
    int32_t strategy;              // pairs: a truncation strategy (PAIR_*, window.cuh) or 0; its rows are written by windows_chunks
    bool dropout;                  // BPE-dropout rows (dropout.cuh), written by windows_chunks: probability, seed, host row keys or NULL
    double drop_p; uint64_t drop_seed; const int64_t* drop_keys;
    genztok_encoded_t* out;
    int32_t old_dirty[4];          // fixed layout: columns of the result planes (ids, mask, token types, sequence ids) that may hold something
                                   // other than padding from the buffer's last use (the width: unknown / a fresh buffer)
};

// The fields genztok_encode and genztok_encode_windows set alike.
EncodeJob make_job(const uint8_t* text, const int64_t* text_off, const uint8_t* pair, const int64_t* pair_off, int32_t max_len, uint32_t flags) {
    EncodeJob J{};
    J.text = text; J.text_off = text_off; J.pair = pair; J.pair_off = pair_off;
    J.max_len = max_len; J.flags = flags;
    J.has_pair = pair_off != nullptr;
    J.want_offs = (flags & GENZTOK_WANT_OFFSETS) != 0;
    J.want_tt = J.has_pair && (flags & GENZTOK_WANT_TOKEN_TYPE);
    J.want_seq = J.has_pair && (flags & GENZTOK_WANT_SEQUENCE_ID);
    return J;
}

// Shard by row across the handle's G devices (SURVEY.md 8e): device g takes the rows [cuts[g], cuts[g + 1]), contiguous ranges
// balanced by weight(r), a non-decreasing prefix over the rows; no collective.  Fewer than two rows per device all go to device 0.
template <class Weight>
std::vector<int64_t> shard_rows(int G, int64_t n, Weight weight) {
    std::vector<int64_t> cuts((size_t)G + 1, n);
    cuts[0] = 0;
    if (G == 1 || n < 2 * G) return cuts;
    const int64_t wtot = weight(n) - weight(0);
    for (int g = 1; g < G; g++) {
        const int64_t want = weight(0) + wtot * g / G;
        int64_t lo = cuts[(size_t)g - 1], hi = n;
        while (lo < hi) { int64_t mid = (lo + hi) / 2; if (weight(mid) < want) lo = mid + 1; else hi = mid; }
        cuts[(size_t)g] = lo;
    }
    return cuts;
}

// work(g) for every device g of the shard cuts: inline when one device has all the rows, else one host thread per device.
template <class Work>
void run_shards(const std::vector<int64_t>& cuts, Work work) {
    const int G = (int)cuts.size() - 1;
    int busy = 0, only = 0;
    for (int g = 0; g < G; g++) if (cuts[(size_t)g + 1] > cuts[(size_t)g]) { busy++; only = g; }
    if (busy <= 1) { work(only); return; }
    std::vector<std::thread> th;
    for (int g = 0; g < G; g++) th.emplace_back([&, g]() { work(g); });
    for (auto& t : th) t.join();
}

// What a device worker reports to the calling thread: its return code, and the text for genztok_last_error.
struct PartStatus {
    int rc = GENZTOK_OK;
    std::string err;
    int report(genztok_t* h) const { std::lock_guard<std::mutex> l(h->err_mu); h->err = err; return rc; }
};

// Failure exits of a device worker, which returns void and has `h`, its stream `st` and its `part` in scope: the part's status is set
// and the stream drained before it returns.  FAIL_RC takes the text that a failed helper left in h->err.
#define PFAIL(code, ...) { char _b[400]; snprintf(_b, sizeof _b, __VA_ARGS__); part->status.rc = (code); part->status.err = _b; cudaStreamSynchronize(st); return; }
#define FAIL_RC(call) { int _rc = (call); if (_rc) { part->status.rc = _rc; { std::lock_guard<std::mutex> _l(h->err_mu); part->status.err = h->err; } cudaStreamSynchronize(st); return; } }
#define CUF(call) { cudaError_t _e = (call); if (_e != cudaSuccess) PFAIL(GENZTOK_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__) }

// Grows a part's array to m entries.  On the part's first chunk of several, `first` is the estimate for the whole part, reserved
// beforehand so that later chunks do not move the array (0: nothing to reserve).
template <class T>
bool grow(PinnedVec<T>& v, size_t m, size_t first) { return (first == 0 || v.reserve(first)) && v.resize(m); }

struct EncodePart {
    PartStatus status;
    int32_t extent = 0;            // fixed layout: columns that can differ from padding, max over this part's chunks
    int64_t d2h_bytes = 0;
    PinnedVec<int32_t> ids, spans, tok_offs; PinnedVec<uint8_t> mask; PinnedVec<int8_t> tt, seq;
    PinnedVec<int64_t> offs, soffs;   // a chunk's row / span offsets on their way home (pinned: a copy into pageable memory is staged by the driver)
    int64_t total = 0, span_total = 0, tokens = 0;
    void bind(genztok_t* h) { ids.h = h; spans.h = h; tok_offs.h = h; mask.h = h; tt.h = h; seq.h = h; offs.h = h; soffs.h = h; }
};

// Chunk boundaries of rows [rb, re): rows [cuts[i], cuts[i+1]) with at most chunk_rows rows and max_chunk_bytes bytes; *most = the
// largest chunk's bytes.  Returns -1, or a document that alone is larger than max_chunk_bytes.
int64_t chunk_cuts(const genztok_t* h, const EncodeJob& J, int64_t rb, int64_t re, std::vector<int64_t>* cuts, int64_t* most) {
    auto bytes_of = [&](int64_t a, int64_t b) { return (J.text_off[b] - J.text_off[a]) + (J.has_pair ? J.pair_off[b] - J.pair_off[a] : 0) + 64; };
    cuts->assign(1, rb);
    *most = 0;
    int64_t r0 = rb;
    while (r0 < re) {
        int64_t r1 = std::min<int64_t>(re, r0 + h->chunk_rows);
        if (bytes_of(r0, r1) > h->max_chunk_bytes) {
            int64_t lo = r0 + 1, hi = r1;   // largest r1 that fits (at least one row)
            while (lo < hi) { int64_t mid = (lo + hi + 1) / 2; if (bytes_of(r0, mid) <= h->max_chunk_bytes) lo = mid; else hi = mid - 1; }
            r1 = lo;
            if (bytes_of(r0, r1) > h->max_chunk_bytes) return r0;
        }
        cuts->push_back(r1);
        *most = std::max<int64_t>(*most, bytes_of(r0, r1));
        r0 = r1;
    }
    return -1;
}

// The rows [r0, r1) of both sides to the device on stream st, into text / toff (and pair / poff), which the caller has sized; *a and
// *b are the sides the kernels read.  Offsets stay absolute (as in the caller's buffer): a side's bytes are copied to dev + (off[r0] & 15)
// and its base pointer is shifted by -off[r0], so that base + 16k is 16-byte aligned, as the kernels' 16-byte loads need.
cudaError_t upload_chunk(const EncodeJob& J, int64_t r0, int64_t r1, DevBuf& text, DevBuf& toff, DevBuf& pair, DevBuf& poff, cudaStream_t st,
                         Side* a, Side* b) {
    auto side = [&](const uint8_t* src, const int64_t* off, DevBuf& bytes, DevBuf& offs, Side* s) {
        const int64_t b0 = off[r0], nb = off[r1] - b0;
        *s = Side{bytes.as<uint8_t>() + (b0 & 15) - b0, offs.as<int64_t>(), nb};
        cudaError_t e = nb ? cudaMemcpyAsync(bytes.as<uint8_t>() + (b0 & 15), src + b0, (size_t)nb, cudaMemcpyHostToDevice, st) : cudaSuccess;
        return e != cudaSuccess ? e : cudaMemcpyAsync(offs.p, off + r0, (size_t)(r1 - r0 + 1) * 8, cudaMemcpyHostToDevice, st);
    };
    *b = Side{nullptr, poff.as<int64_t>(), 0};
    cudaError_t e = side(J.text, J.text_off, text, toff, a);
    return (e != cudaSuccess || !J.has_pair) ? e : side(J.pair, J.pair_off, pair, poff, b);
}

// The devices' rows of a host-buffer encode or windows call, part g on device g: the frame around chunks(d, cuts, part), which issues
// the chunks of the part's rows on d->stream and leaves a failure in the part's status.  A part is ordered behind the previous user of
// the device context's shared work areas (stream_enter) before anything touches them; the word cache is sized for its largest chunk;
// the token and error counters are read around its chunks.
template <class Part, class Chunks>
void run_parts(genztok_t* h, const EncodeJob& J, const std::vector<int64_t>& dcut, std::vector<Part>& parts, Chunks chunks) {
    for (auto& pt : parts) pt.bind(h);
    run_shards(dcut, [&](int g) {
        DeviceCtx* d = h->devs[(size_t)g];
        Part* part = &parts[(size_t)g];
        cudaStream_t st = d->stream;
        CUF(cudaSetDevice(d->device));
        LaunchScope::cur_stream = st;
        FAIL_RC(stream_enter(h, d, st));
        std::vector<int64_t> cuts;
        int64_t most = 0;
        { const int64_t big = chunk_cuts(h, J, dcut[(size_t)g], dcut[(size_t)g + 1], &cuts, &most);
          if (big >= 0) PFAIL(GENZTOK_E_LIMIT, "document %lld is larger than max_chunk_bytes=%lld", (long long)big, (long long)h->max_chunk_bytes) }
        FAIL_RC(ensure_cache(h, d, st, most));
        if (J.want_offs) FAIL_RC(ensure_piece_lens(h, d, st));
        unsigned long long tokens_before = 0, tokens_after = 0, nerr = 0;
        CUF(cudaMemcpyAsync(&tokens_before, d->C.ctr + C_TOKENS, 8, cudaMemcpyDeviceToHost, st));
        CUF(cudaStreamSynchronize(st));
        chunks(d, cuts, part);
        if (part->status.rc) return;
        CUF(cudaMemcpyAsync(&tokens_after, d->C.ctr + C_TOKENS, 8, cudaMemcpyDeviceToHost, st));
        CUF(cudaMemcpyAsync(&nerr, d->C.ctr + C_ERR, 8, cudaMemcpyDeviceToHost, st));
        CUF(cudaStreamSynchronize(st));
        if (nerr) PFAIL(GENZTOK_E_CUDA, "internal error: device pipeline reported %llu inconsistencies", nerr)
        part->tokens = (int64_t)(tokens_after - tokens_before);
        FAIL_RC(stream_leave(h, d, st));
    });
}

// Fixed layout, pipelined over chunks: H2D(i + 1) | kernels(i) | D2H(i - 1) on three streams, two sets of chunk buffers.
// Only the columns that can differ from padding travel back: [0, max(extent of the chunk, what the pooled host plane still
// holds from its last use)), rounded up to 32; a fresh host plane takes whole rows once.
void encode_fixed_chunks(genztok_t* h, DeviceCtx* d, const EncodeJob& J, const std::vector<int64_t>& cuts, EncodePart* part) {
    cudaStream_t st = d->stream;
    genztok_encoded_t* out = J.out;
    const bool has_pair = J.has_pair, want_tt = J.want_tt, want_seq = J.want_seq;
    const int32_t max_len = J.max_len;
    const size_t nc = cuts.size() - 1;
    if (!d->s_in) CUF(cudaStreamCreateWithFlags(&d->s_in, cudaStreamNonBlocking));
    if (!d->s_out) CUF(cudaStreamCreateWithFlags(&d->s_out, cudaStreamNonBlocking));
    if (!d->h_extent) CUF(cudaHostAlloc(reinterpret_cast<void**>(&d->h_extent), 64, cudaHostAllocDefault));
    int64_t mm = 0, mtb = 0, mpb = 0;
    for (size_t ci = 0; ci < nc; ci++) {
        mm = std::max(mm, cuts[ci + 1] - cuts[ci]);
        mtb = std::max(mtb, J.text_off[cuts[ci + 1]] - J.text_off[cuts[ci]]);
        if (has_pair) mpb = std::max(mpb, J.pair_off[cuts[ci + 1]] - J.pair_off[cuts[ci]]);
    }
    const size_t mtot = (size_t)mm * (size_t)max_len;
    for (int sidx = 0; sidx < (nc > 1 ? 2 : 1); sidx++) {
        DeviceCtx::Stage& sg = d->stage[sidx];
        for (cudaEvent_t* e : {&sg.h2d, &sg.k, &sg.d2h}) if (!*e) CUF(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        CUF(sg.text.ensure((size_t)mtb + 96)); CUF(sg.toff.ensure((size_t)(mm + 1) * 8));
        if (has_pair) { CUF(sg.pair.ensure((size_t)mpb + 96)); CUF(sg.poff.ensure((size_t)(mm + 1) * 8)); }
        CUF(sg.ids.ensure(mtot * 4)); CUF(sg.mask.ensure(mtot)); CUF(sg.row_len.ensure((size_t)mm * 4)); CUF(sg.extent.ensure(16));
        if (want_tt) CUF(sg.tt.ensure(mtot));
        if (want_seq) CUF(sg.seq.ensure(mtot));
        if (has_pair) { CUF(sg.seq_len.ensure((size_t)mm * 4)); CUF(sg.status.ensure((size_t)mm)); }
    }
    Side in_a[2], in_b[2];                                            // the sides of the chunks in the two sets
    auto issue_h2d = [&](size_t ci) -> bool {
        DeviceCtx::Stage& sg = d->stage[ci & 1];
        if (ci >= 2 && cudaStreamWaitEvent(d->s_in, sg.k, 0) != cudaSuccess) return false;      // the kernels of chunk ci - 2 have read this set's inputs
        if (upload_chunk(J, cuts[ci], cuts[ci + 1], sg.text, sg.toff, sg.pair, sg.poff, d->s_in, &in_a[ci & 1], &in_b[ci & 1]) != cudaSuccess) return false;
        return cudaEventRecord(sg.h2d, d->s_in) == cudaSuccess;
    };
    auto fail_sync = [&]() { cudaStreamSynchronize(d->s_in); cudaStreamSynchronize(st); cudaStreamSynchronize(d->s_out); };
    if (nc && !issue_h2d(0)) { fail_sync(); PFAIL(GENZTOK_E_CUDA, "host to device copy failed: %s", cudaGetErrorString(cudaGetLastError())) }
    for (size_t ci = 0; ci < nc; ci++) {
        DeviceCtx::Stage& sg = d->stage[ci & 1];
        const int64_t r0 = cuts[ci], r1 = cuts[ci + 1], m = r1 - r0;
        // kernels of chunk ci: behind its inputs, and behind the copy-out of the chunk that used this set of planes before
        CUF(cudaStreamWaitEvent(st, sg.h2d, 0));
        if (ci >= 2) CUF(cudaStreamWaitEvent(st, sg.d2h, 0));
        genztok_dev_planes_t P{};
        P.input_ids = sg.ids.as<int32_t>(); P.attention_mask = sg.mask.as<uint8_t>(); P.row_len = sg.row_len.as<int32_t>();
        if (want_tt) P.token_type_ids = sg.tt.as<int8_t>();
        if (want_seq) P.sequence_id = sg.seq.as<int8_t>();
        if (has_pair) { P.seq_len = sg.seq_len.as<int32_t>(); P.row_status = sg.status.as<uint8_t>(); }
        if (int rc = encode_fixed_on_device(h, d, st, in_a[ci & 1], has_pair ? &in_b[ci & 1] : nullptr, m, max_len, J.flags, P)) { fail_sync(); FAIL_RC(rc) }
        CUF(cudaMemsetAsync(sg.extent.p, 0, 4, st));
        { LaunchScope ls(h, d, "k_row_extent");
          k_row_extent<<<(unsigned)std::min<int64_t>((m + 255) / 256, (int64_t)d->sm_count * 4), 256, 0, st>>>(P.row_len, has_pair ? P.seq_len : nullptr, m, sg.extent.as<int32_t>()); }
        CUF(cudaMemcpyAsync(d->h_extent + (ci & 1), sg.extent.p, 4, cudaMemcpyDeviceToHost, st));
        CUF(cudaEventRecord(sg.k, st));
        // the next chunk's inputs travel while these kernels run
        if (ci + 1 < nc && !issue_h2d(ci + 1)) { fail_sync(); PFAIL(GENZTOK_E_CUDA, "host to device copy failed: %s", cudaGetErrorString(cudaGetLastError())) }
        // copy-out of chunk ci: the host learns the extent (the only wait of this loop), then the trimmed planes go on their own stream
        CUF(cudaEventSynchronize(sg.k));
        const int32_t kc = std::min<int32_t>(max_len, std::max<int32_t>(d->h_extent[ci & 1], 1));
        part->extent = std::max(part->extent, kc);
        CUF(cudaStreamWaitEvent(d->s_out, sg.k, 0));
        const size_t o0 = (size_t)r0 * (size_t)max_len;
        CopyOutArgs CO{};
        CO.m = m;
        auto copy_plane = [&](void* host, const void* dev, size_t elt, int32_t old_dirty) -> cudaError_t {
            // whole 64-byte lines of host memory for the one-byte planes too (a partial line is a read-modify-write for the host)
            const int32_t rnd = elt == 1 ? (int32_t)std::max<int64_t>(32, h->copy_round) : 32;
            const int32_t cols = std::min<int32_t>(max_len, (std::max(kc, old_dirty) + rnd - 1) / rnd * rnd);
            part->d2h_bytes += (int64_t)m * cols * (int64_t)elt;
            uint8_t* dst = reinterpret_cast<uint8_t*>(host) + o0 * elt;
            if (cols >= max_len) return cudaMemcpyAsync(dst, dev, (size_t)m * (size_t)max_len * elt, cudaMemcpyDeviceToHost, d->s_out);
            void* dmap = nullptr;                                     // trimmed rows: stores of a kernel into the mapped host plane
            if (!h->no_copy_kernel && ((size_t)max_len * elt) % 16 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0 &&
                cudaHostGetDevicePointer(&dmap, dst, 0) == cudaSuccess && dmap) {
                CO.p[CO.n_planes++] = CopyOutPlane{reinterpret_cast<const uint8_t*>(dev), reinterpret_cast<uint8_t*>(dmap), (uint32_t)(max_len * elt), (uint32_t)(cols * elt)};
                return cudaSuccess;
            }
            cudaGetLastError();
            return cudaMemcpy2DAsync(dst, (size_t)max_len * elt, dev, (size_t)max_len * elt, (size_t)cols * elt, (size_t)m, cudaMemcpyDeviceToHost, d->s_out);
        };
        CUF(copy_plane(out->input_ids, sg.ids.p, 4, J.old_dirty[0]));
        CUF(copy_plane(out->attention_mask, sg.mask.p, 1, J.old_dirty[1]));
        if (want_tt) CUF(copy_plane(out->token_type_ids, sg.tt.p, 1, J.old_dirty[2]));
        if (want_seq) CUF(copy_plane(out->sequence_id, sg.seq.p, 1, J.old_dirty[3]));
        if (CO.n_planes) {
            LaunchScope::cur_stream = d->s_out;
            { LaunchScope ls(h, d, "k_copy_out"); k_copy_out<<<(unsigned)std::max<int64_t>(1, h->copy_blocks), 256, 0, d->s_out>>>(CO); }
            LaunchScope::cur_stream = st;
            CUF(cudaGetLastError());
        }
        CUF(cudaMemcpyAsync(out->row_len + r0, sg.row_len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, d->s_out));
        part->d2h_bytes += m * 4;
        if (has_pair) {
            CUF(cudaMemcpyAsync(out->seq_len + r0, sg.seq_len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, d->s_out));
            CUF(cudaMemcpyAsync(out->row_status + r0, sg.status.p, (size_t)m, cudaMemcpyDeviceToHost, d->s_out));
            part->d2h_bytes += m * 5;
        }
        CUF(cudaEventRecord(sg.d2h, d->s_out));
    }
    CUF(cudaStreamSynchronize(d->s_out));
}

// Ragged layout, chunk after chunk on d->stream: the planes come home into the part's pinned arrays, row offsets relative to the part.
void encode_ragged_chunks(genztok_t* h, DeviceCtx* d, const EncodeJob& J, const std::vector<int64_t>& cuts, EncodePart* part) {
    cudaStream_t st = d->stream;
    genztok_encoded_t* out = J.out;
    const bool has_pair = J.has_pair, has_max_len = J.has_max_len, want_spans = J.want_spans;
    const int32_t max_len = J.max_len;
    const int8_t eos8 = eos_as_i8(d);
    const int64_t rb = cuts.front(), re = cuts.back();
    for (size_t ci = 0; ci + 1 < cuts.size(); ci++) {
        const int64_t r0 = cuts[ci], r1 = cuts[ci + 1], m = r1 - r0;
        const int64_t tb = J.text_off[r1] - J.text_off[r0], pb = has_pair ? J.pair_off[r1] - J.pair_off[r0] : 0;
        CUF(d->text.ensure((size_t)tb + 96)); CUF(d->toff.ensure((size_t)(m + 1) * 8));
        if (has_pair) { CUF(d->pair.ensure((size_t)pb + 96)); CUF(d->poff.ensure((size_t)(m + 1) * 8)); }
        Side a, b;
        CUF(upload_chunk(J, r0, r1, d->text, d->toff, d->pair, d->poff, st, &a, &b));
        CUF(d->redo.ensure((size_t)m * 4)); CUF(d->fix.ensure((size_t)m * 4));
        CUF(d->L.ensure((size_t)m * 4)); CUF(d->keep.ensure((size_t)m * 4)); CUF(d->out_len.ensure((size_t)m * 8));
        CUF(d->row_off.ensure((size_t)(m + 1) * 8)); CUF(d->tail.ensure((size_t)m));
        FAIL_RC(launch_guard(h, d, st, tb + pb + 16, 0));
        RowArgs A{};
        A.a = a; A.b = b; A.has_pair = has_pair; A.n_rows = m; A.W = 0; A.flags = J.flags;
        A.L = d->L.as<int32_t>(); A.redo_list = d->redo.as<uint32_t>(); A.fix_list = d->fix.as<uint32_t>(); A.eos_i8 = eos8; A.pad_i8 = pad_as_i8(d);
        if (want_spans) {
            CUF(d->nwA.ensure((size_t)m * 4)); CUF(d->nwB.ensure((size_t)m * 4)); CUF(d->span_cnt.ensure((size_t)m * 8)); CUF(d->span_off.ensure((size_t)(m + 1) * 8));
            A.nwA = d->nwA.as<int32_t>(); A.nwB = d->nwB.as<int32_t>();
        }
        A.D = pick_tile_docs(h, d, tb, pb, m, 0, false);
        FAIL_RC(launch_rows<MODE_COUNT>(h, d, A, st, "k_rows_count", m));
        FAIL_RC(launch_bpe(h, d, st));
        RowArgs R = A; R.row_list = d->redo.as<uint32_t>();
        FAIL_RC(launch_rows<MODE_COUNT>(h, d, R, st, "k_rows_count_redo", std::min<int64_t>(m, (int64_t)d->sm_count * 64)));
        LenArgs LA{d->L.as<int32_t>(), m, (int32_t)has_max_len, has_max_len ? max_len : 0, J.padding ? 1 : 0, J.truncation ? 1 : 0,
                   d->keep.as<int32_t>(), d->out_len.as<int64_t>(), d->tail.as<uint8_t>(),
                   want_spans ? d->nwA.as<int32_t>() : nullptr, (want_spans && has_pair) ? d->nwB.as<int32_t>() : nullptr,
                   want_spans ? d->span_cnt.as<int64_t>() : nullptr};
        { LaunchScope ls(h, d, "k_row_lens"); k_row_lens<<<(unsigned)std::min<int64_t>((m + 255) / 256, 4096), 256, 0, st>>>(LA); }
        FAIL_RC(launch_scan(h, d, st, d->out_len.as<int64_t>(), d->row_off.as<int64_t>(), m));
        int64_t total = 0, span_n = 0;
        if (want_spans) {
            FAIL_RC(launch_scan(h, d, st, d->span_cnt.as<int64_t>(), d->span_off.as<int64_t>(), m));
            CUF(cudaMemcpyAsync(&span_n, d->span_off.as<int64_t>() + m, 8, cudaMemcpyDeviceToHost, st));
        }
        CUF(cudaMemcpyAsync(&total, d->row_off.as<int64_t>() + m, 8, cudaMemcpyDeviceToHost, st));
        CUF(cudaStreamSynchronize(st));
        if (want_spans) CUF(d->spans.ensure((size_t)span_n * 8 + 16));
        CUF(d->ids.ensure((size_t)total * 4 + 16)); CUF(d->mask.ensure((size_t)total + 16)); CUF(d->row_len.ensure((size_t)m * 4));
        if (has_pair) { CUF(d->tt.ensure((size_t)total + 16)); CUF(d->seq.ensure((size_t)total + 16)); CUF(d->seq_len.ensure((size_t)m * 4)); CUF(d->tt_len.ensure((size_t)m * 4)); CUF(d->status.ensure((size_t)m)); }
        { LaunchScope ls(h, d, "k_reset_lists"); k_reset_lists<<<1, 1, 0, st>>>(d->C); }
        RowArgs E = A;
        E.ids = d->ids.as<int32_t>(); E.row_off = d->row_off.as<int64_t>(); E.keep = d->keep.as<int32_t>();
        if (want_spans) { E.span_off = d->span_off.as<int64_t>(); E.spans = d->spans.as<int32_t>(); }
        if (J.want_offs) {                                          // framing, pads and a forced </s> keep the (0, 0) of the memset
            CUF(d->offs.ensure((size_t)total * 8 + 16));
            CUF(cudaMemsetAsync(d->offs.p, 0, (size_t)total * 8, st));
            E.offs = d->offs.as<int32_t>(); E.plen = d->len_arena.as<uint16_t>();
        }
        FAIL_RC(launch_rows<MODE_RAGGED>(h, d, E, st, J.want_offs ? "k_rows_ragged_offsets" : "k_rows_ragged", m));
        PostArgs Q{};
        Q.ids = d->ids.as<int32_t>(); Q.row_off = d->row_off.as<int64_t>(); Q.n_rows = m; Q.keep = d->keep.as<int32_t>(); Q.tail = d->tail.as<uint8_t>();
        Q.mask = d->mask.as<uint8_t>(); Q.has_pair = has_pair; Q.row_len = d->row_len.as<int32_t>();
        if (has_pair) { Q.tt = d->tt.as<int8_t>(); Q.seq = d->seq.as<int8_t>(); Q.tt_len = d->tt_len.as<int32_t>(); Q.seq_len = d->seq_len.as<int32_t>(); Q.status = d->status.as<uint8_t>(); }
        Q.has_max_len = has_max_len; Q.max_len = has_max_len ? max_len : 0; Q.padding = J.padding ? 1 : 0; Q.truncation = J.truncation ? 1 : 0; Q.eos_i8 = eos8; Q.pad_i8 = pad_as_i8(d);
        Q.tokens_ctr = d->C.ctr + C_TOKENS;
        { LaunchScope ls(h, d, "k_post_rows"); k_post_rows<<<(unsigned)std::min<int64_t>((m + 7) / 8, (int64_t)d->sm_count * 8), 256, 0, st>>>(d->T, Q, nullptr); }
        CUF(cudaGetLastError());
        // bring the chunk home; offsets are kept relative to this device's part
        const size_t old = part->ids.size(), nt = old + (size_t)total;
        // first chunk of several: room for the whole part at this chunk's tokens per row (+ 12 %)
        const size_t est = (old == 0 && r1 < re) ? (size_t)((double)total * (double)(re - rb) / (double)m * 1.125) + 4096 : 0;
        bool grown = grow(part->ids, nt, est) && grow(part->mask, nt, est);
        if (has_pair) grown = grown && grow(part->tt, nt, est) && grow(part->seq, nt, est);
        if (J.want_offs) grown = grown && grow(part->tok_offs, 2 * nt, 2 * est);
        grown = grown && part->offs.resize((size_t)m + 1);
        if (!grown) PFAIL(GENZTOK_E_NOMEM, "pinned host allocation failed")
        int64_t* const offs = part->offs.data();
        if (total) {
            CUF(cudaMemcpyAsync(part->ids.data() + old, d->ids.p, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
            CUF(cudaMemcpyAsync(part->mask.data() + old, d->mask.p, (size_t)total, cudaMemcpyDeviceToHost, st));
            if (has_pair) {
                CUF(cudaMemcpyAsync(part->tt.data() + old, d->tt.p, (size_t)total, cudaMemcpyDeviceToHost, st));
                CUF(cudaMemcpyAsync(part->seq.data() + old, d->seq.p, (size_t)total, cudaMemcpyDeviceToHost, st));
            }
            if (J.want_offs) CUF(cudaMemcpyAsync(part->tok_offs.data() + 2 * old, d->offs.p, (size_t)total * 8, cudaMemcpyDeviceToHost, st));
        }
        int64_t* soffs = nullptr;
        if (want_spans) {
            if (!part->soffs.resize((size_t)m + 1)) PFAIL(GENZTOK_E_NOMEM, "pinned host allocation failed")
            soffs = part->soffs.data();
            const size_t so = part->spans.size();
            if (so == 0 && r1 < re && !part->spans.reserve((size_t)((double)span_n * 2.0 * (double)(re - rb) / (double)m * 1.125) + 4096)) PFAIL(GENZTOK_E_NOMEM, "pinned host allocation failed")
            if (!part->spans.resize(so + (size_t)span_n * 2)) PFAIL(GENZTOK_E_NOMEM, "pinned host allocation failed")
            if (span_n) CUF(cudaMemcpyAsync(part->spans.data() + so, d->spans.p, (size_t)span_n * 8, cudaMemcpyDeviceToHost, st));
            CUF(cudaMemcpyAsync(soffs, d->span_off.p, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
        }
        CUF(cudaMemcpyAsync(offs, d->row_off.p, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
        CUF(cudaMemcpyAsync(out->row_len + r0, d->row_len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
        if (has_pair) {
            CUF(cudaMemcpyAsync(out->seq_len + r0, d->seq_len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
            CUF(cudaMemcpyAsync(out->tt_len + r0, d->tt_len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
            CUF(cudaMemcpyAsync(out->row_status + r0, d->status.p, (size_t)m, cudaMemcpyDeviceToHost, st));
        }
        CUF(cudaStreamSynchronize(st));
        part->d2h_bytes += total * (has_pair ? 7 : 5) + (m + 1) * 8 + m * (has_pair ? 13 : 4) + (want_spans ? span_n * 8 + (m + 1) * 8 : 0) + (J.want_offs ? total * 8 : 0);
        for (int64_t i = 1; i <= m; i++) out->row_off[r0 + i] = part->total + offs[i];      // relative to the part
        part->total += total;
        if (want_spans) { for (int64_t i = 1; i <= m; i++) out->span_off[r0 + i] = part->span_total + soffs[i]; part->span_total += span_n; }
    }
}

// What one device collects for its documents [rb, re) of genztok_encode_windows (chunk after chunk, in document order).
struct WindowPart {
    PartStatus status;
    int64_t n_win = 0, tokens = 0, d2h_bytes = 0;
    PinnedVec<int32_t> ids, row_len, seq_len, start, tok_offs; PinnedVec<uint8_t> mask, row_status; PinnedVec<int8_t> tt, seq; PinnedVec<int64_t> doc, offs;
    void bind(genztok_t* h) { for (auto* v : {&ids, &row_len, &seq_len, &start, &tok_offs}) v->h = h; mask.h = h; row_status.h = h; tt.h = h; seq.h = h; doc.h = h; offs.h = h; }
};

// Windows of one device's chunks: per chunk the text goes up, both steps run, the planes and maps come home.
// win_off[r] for r in (rb, re] is written relative to the part's first window.
// With J.strategy or J.dropout the chunk's rows (one per document) go straight into the fixed-layout planes of J.out at their rows,
// and win_off is not used.
void windows_chunks(genztok_t* h, DeviceCtx* d, const EncodeJob& J, int32_t stride, int64_t* win_off, const std::vector<int64_t>& cuts, WindowPart* part) {
    cudaStream_t st = d->stream;
    const bool has_pair = J.has_pair, rows = J.strategy != 0 || J.dropout;
    const int32_t W = J.max_len;
    const int64_t rb = cuts.front(), re = cuts.back();
    for (size_t ci = 0; ci + 1 < cuts.size(); ci++) {
        const int64_t r0 = cuts[ci], r1 = cuts[ci + 1], m = r1 - r0;
        const int64_t tb = J.text_off[r1] - J.text_off[r0], pb = has_pair ? J.pair_off[r1] - J.pair_off[r0] : 0;
        CUF(d->text.ensure((size_t)tb + 96)); CUF(d->toff.ensure((size_t)(m + 1) * 8));
        if (has_pair) { CUF(d->pair.ensure((size_t)pb + 96)); CUF(d->poff.ensure((size_t)(m + 1) * 8)); }
        Side a, b;
        CUF(upload_chunk(J, r0, r1, d->text, d->toff, d->pair, d->poff, st, &a, &b));
        CUF(d->win.woff.ensure((size_t)(m + 1) * 8));
        int64_t K = m;
        if (J.dropout) {                                             // the row keys: the caller's, or the rows' indices in the whole call
            const int64_t* keys = nullptr;
            if (J.drop_keys) {
                CUF(d->win.drop_keys.ensure((size_t)m * 8));
                CUF(cudaMemcpyAsync(d->win.drop_keys.p, J.drop_keys + r0, (size_t)m * 8, cudaMemcpyHostToDevice, st));
                keys = d->win.drop_keys.as<int64_t>();
            }
            FAIL_RC(dropout_layout(h, d, st, a, has_pair ? &b : nullptr, m, W, J.drop_p, J.drop_seed, keys, r0));
        } else {
            FAIL_RC(windows_layout(h, d, st, a, has_pair ? &b : nullptr, m, W, stride, J.strategy, J.want_offs, d->win.woff.as<int64_t>(), &K));
        }
        const size_t tot = (size_t)K * (size_t)W;
        CUF(d->ids.ensure(tot * 4 + 16)); CUF(d->mask.ensure(tot + 16)); CUF(d->row_len.ensure((size_t)K * 4 + 16));
        CUF(d->win.doc.ensure((size_t)K * 8 + 16)); CUF(d->win.start.ensure((size_t)K * 4 + 16));
        genztok_dev_planes_t P{};
        P.input_ids = d->ids.as<int32_t>(); P.attention_mask = d->mask.as<uint8_t>(); P.row_len = d->row_len.as<int32_t>();
        if (J.want_tt) { CUF(d->tt.ensure(tot + 16)); P.token_type_ids = d->tt.as<int8_t>(); }
        if (J.want_seq) { CUF(d->seq.ensure(tot + 16)); P.sequence_id = d->seq.as<int8_t>(); }
        if (has_pair) { CUF(d->seq_len.ensure((size_t)K * 4 + 16)); CUF(d->status.ensure((size_t)K + 16)); P.seq_len = d->seq_len.as<int32_t>(); P.row_status = d->status.as<uint8_t>(); }
        if (J.want_offs) { CUF(d->win.plane_offs.ensure(tot * 8 + 16)); P.offsets = d->win.plane_offs.as<int32_t>(); }
        FAIL_RC(windows_write(h, d, st, has_pair, m, W, stride, J.dropout ? STREAMS_CAPPED : J.strategy, J.flags, d->win.woff.as<int64_t>(), K, P,
                              d->win.doc.as<int64_t>(), d->win.start.as<int32_t>(), r0));
        // where the chunk's rows go on the host: the result planes at rows r0.. (strategy), else the part's arrays behind its windows so far
        genztok_dev_planes_t H{};
        size_t o = (size_t)r0;
        if (rows) {
            const genztok_encoded_t* out = J.out;
            H.input_ids = out->input_ids; H.attention_mask = out->attention_mask; H.token_type_ids = out->token_type_ids; H.sequence_id = out->sequence_id;
            H.row_len = out->row_len; H.seq_len = out->seq_len; H.row_status = out->row_status; H.offsets = out->offsets;
        } else {
            o = (size_t)part->n_win;
            const size_t n1 = o + (size_t)K;
            // first chunk of several: room for the part at this chunk's windows per document (+ 12 %)
            const size_t est = (ci == 0 && r1 < re) ? (size_t)((double)K * (double)(re - rb) / (double)m * 1.125) + 64 : 0;
            bool grown = grow(part->ids, n1 * W, est * W) && grow(part->mask, n1 * W, est * W) && grow(part->row_len, n1, est) && grow(part->doc, n1, est) &&
                         grow(part->start, n1, est) && part->offs.resize((size_t)m + 1);
            if (J.want_tt) grown = grown && grow(part->tt, n1 * W, est * W);
            if (J.want_seq) grown = grown && grow(part->seq, n1 * W, est * W);
            if (J.want_offs) grown = grown && grow(part->tok_offs, 2 * n1 * W, 2 * est * W);
            if (has_pair) grown = grown && grow(part->seq_len, n1, est) && grow(part->row_status, n1, est);
            if (!grown) PFAIL(GENZTOK_E_NOMEM, "pinned host allocation failed")
            H.input_ids = part->ids.data(); H.attention_mask = part->mask.data(); H.token_type_ids = part->tt.data(); H.sequence_id = part->seq.data();
            H.row_len = part->row_len.data(); H.seq_len = part->seq_len.data(); H.row_status = part->row_status.data(); H.offsets = part->tok_offs.data();
        }
        if (K) {
            CUF(cudaMemcpyAsync(H.input_ids + o * W, P.input_ids, tot * 4, cudaMemcpyDeviceToHost, st));
            CUF(cudaMemcpyAsync(H.attention_mask + o * W, P.attention_mask, tot, cudaMemcpyDeviceToHost, st));
            if (J.want_tt) CUF(cudaMemcpyAsync(H.token_type_ids + o * W, P.token_type_ids, tot, cudaMemcpyDeviceToHost, st));
            if (J.want_seq) CUF(cudaMemcpyAsync(H.sequence_id + o * W, P.sequence_id, tot, cudaMemcpyDeviceToHost, st));
            if (J.want_offs) CUF(cudaMemcpyAsync(H.offsets + 2 * o * W, P.offsets, tot * 8, cudaMemcpyDeviceToHost, st));
            CUF(cudaMemcpyAsync(H.row_len + o, P.row_len, (size_t)K * 4, cudaMemcpyDeviceToHost, st));
            if (!rows) {
                CUF(cudaMemcpyAsync(part->doc.data() + o, d->win.doc.p, (size_t)K * 8, cudaMemcpyDeviceToHost, st));
                CUF(cudaMemcpyAsync(part->start.data() + o, d->win.start.p, (size_t)K * 4, cudaMemcpyDeviceToHost, st));
            }
            if (has_pair) {
                CUF(cudaMemcpyAsync(H.seq_len + o, P.seq_len, (size_t)K * 4, cudaMemcpyDeviceToHost, st));
                CUF(cudaMemcpyAsync(H.row_status + o, P.row_status, (size_t)K, cudaMemcpyDeviceToHost, st));
            }
        }
        if (!rows) CUF(cudaMemcpyAsync(part->offs.data(), d->win.woff.p, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
        CUF(cudaStreamSynchronize(st));
        part->d2h_bytes += (int64_t)tot * (5 + (J.want_tt ? 1 : 0) + (J.want_seq ? 1 : 0) + (J.want_offs ? 8 : 0)) + K * (4 + (has_pair ? 5 : 0)) +
                           (rows ? 0 : K * 12 + (m + 1) * 8);
        if (!rows) {
            const int64_t* offs = part->offs.data();
            for (int64_t i = 1; i <= m; i++) win_off[r0 + i] = part->n_win + offs[i];
        }
        part->n_win += K;
    }
}

// BPE-dropout of a host-buffer encode (genztok_encode_dropout): probability, seed, host row keys or NULL.
struct DropSpec { double p; uint64_t seed; const int64_t* keys; };

int encode_host(genztok_t* h, const uint8_t* text, const int64_t* text_off, const uint8_t* pair, const int64_t* pair_off, int64_t n, int32_t max_len,
                int padding, int truncation, uint32_t flags, int32_t strategy, const DropSpec* drop, genztok_encoded_t* out);

}  // namespace

extern "C" {

int genztok_encode(genztok_t* h, const uint8_t* text, const int64_t* text_off, const uint8_t* pair, const int64_t* pair_off, int64_t n,
                   int32_t max_len, int padding, int truncation, uint32_t flags, genztok_encoded_t* out) {
    if (!h) return GENZTOK_E_INVALID;
    if (!out || n < 0 || !text_off) return fail(h, GENZTOK_E_INVALID, "genztok_encode: bad arguments");
    int32_t strategy = 0;
    { const int rc = pair_strategy(h, flags, max_len, padding && truncation && !(flags & GENZTOK_WANT_SPANS), &strategy); if (rc) return rc; }
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    return encode_host(h, text, text_off, pair, pair_off, n, max_len, padding, truncation, flags, strategy, nullptr, out);
}

}  // extern "C"

namespace {

// The host-buffer encode after its argument checks.  drop: the rows of BPE-dropout (the fixed layout, the reference cut), written by
// windows_chunks like those of a truncation strategy.
int encode_host(genztok_t* h, const uint8_t* text, const int64_t* text_off, const uint8_t* pair, const int64_t* pair_off, int64_t n, int32_t max_len,
                int padding, int truncation, uint32_t flags, int32_t strategy, const DropSpec* drop, genztok_encoded_t* out) {
    memset(out, 0, sizeof *out);
    std::lock_guard<std::mutex> lk(h->mu);
    EncodeJob J = make_job(text, text_off, pair, pair_off, max_len, flags);
    J.padding = padding; J.truncation = truncation; J.out = out;
    J.has_max_len = max_len != GENZTOK_MAX_LEN_NONE;
    J.want_spans = (flags & GENZTOK_WANT_SPANS) != 0;       // return_offset: produced by the ragged pipeline
    J.strategy = J.has_pair ? strategy : 0;                 // (without second texts every strategy is the reference cut)
    if (drop) { J.dropout = true; J.drop_p = drop->p; J.drop_seed = drop->seed; J.drop_keys = drop->keys; }
    const bool rows = J.strategy || J.dropout;              // one row per document from windows_chunks
    // the fixed regime; with offsets (offset_mapping) it is computed by the ragged pipeline, whose rows then all hold max_len
    // entries, and presented in the fixed layout; the rows of a truncation strategy or of BPE-dropout are written by windows_chunks
    const bool fixed_layout = J.has_max_len && max_len >= 1 && padding && truncation && (rows || fixed_fits(h->devs[0], max_len)) && !J.want_spans;
    J.fixed = fixed_layout && !J.want_offs && !rows;
    const bool has_pair = J.has_pair, fixed = J.fixed;
    OutBlock* ob = new OutBlock();
    out->_owner = ob;
    out->n = n; out->has_pair = has_pair;
    auto free_nolock = [&]() { discard_block(h, ob); memset(out, 0, sizeof *out); };
    // offsets in the fixed regime: every row of the ragged result is a padded / truncated row of max_len entries
    auto present_fixed = [&]() -> int {
        if (out->row_off[n] != n * (int64_t)max_len) {
            free_nolock();
            return fail(h, GENZTOK_E_CUDA, "internal error: fixed-regime rows do not hold max_len entries");
        }
        out->width = max_len; out->row_off = nullptr;
        if (!J.want_tt) { out->token_type_ids = nullptr; out->tt_len = nullptr; }   // the planes the fixed layout leaves out
        if (!J.want_seq) out->sequence_id = nullptr;
        return GENZTOK_OK;
    };
#define OOM_CHECK(p) if (!(p)) { free_nolock(); return fail(h, GENZTOK_E_NOMEM, "pinned host allocation failed"); }
    if (J.want_spans) { out->span_off = out_alloc<int64_t>(h, ob, (size_t)n + 1); OOM_CHECK(out->span_off); out->span_off[0] = 0; }
    if (fixed || rows) {
        const size_t tot = (size_t)n * (size_t)max_len;
        out->width = max_len; out->total = (int64_t)tot;
        out->input_ids = out_alloc<int32_t>(h, ob, tot); OOM_CHECK(out->input_ids);
        out->attention_mask = out_alloc<uint8_t>(h, ob, tot); OOM_CHECK(out->attention_mask);
        out->row_len = out_alloc<int32_t>(h, ob, (size_t)n); OOM_CHECK(out->row_len);
        if (J.want_tt) { out->token_type_ids = out_alloc<int8_t>(h, ob, tot); OOM_CHECK(out->token_type_ids); out->tt_len = out_alloc<int32_t>(h, ob, (size_t)n); OOM_CHECK(out->tt_len); }
        if (J.want_seq) { out->sequence_id = out_alloc<int8_t>(h, ob, tot); OOM_CHECK(out->sequence_id); }
        if (has_pair) { out->seq_len = out_alloc<int32_t>(h, ob, (size_t)n); OOM_CHECK(out->seq_len); out->row_status = out_alloc<uint8_t>(h, ob, (size_t)n); OOM_CHECK(out->row_status); }
        if (rows) {
            if (J.want_offs) { out->offsets = out_alloc<int32_t>(h, ob, 2 * tot); OOM_CHECK(out->offsets); }
            for (auto& pr : ob->pinned) h->plane_meta.erase(pr.first);   // (these planes are written whole; no record describes them)
        }
    } else {
        out->width = 0;
        out->row_off = out_alloc<int64_t>(h, ob, (size_t)n + 1); OOM_CHECK(out->row_off);
        out->row_len = out_alloc<int32_t>(h, ob, (size_t)n); OOM_CHECK(out->row_len);
        if (has_pair) {
            out->seq_len = out_alloc<int32_t>(h, ob, (size_t)n); OOM_CHECK(out->seq_len);
            out->tt_len = out_alloc<int32_t>(h, ob, (size_t)n); OOM_CHECK(out->tt_len);
            out->row_status = out_alloc<uint8_t>(h, ob, (size_t)n); OOM_CHECK(out->row_status);
        }
        out->row_off[0] = 0;
    }
#undef OOM_CHECK
    // what the pooled planes still hold from their last use (see encode_rows_on_device, fixed layout)
    void* const planes4[4] = {out->input_ids, out->attention_mask, out->token_type_ids, out->sequence_id};
    const int32_t elts4[4] = {4, 1, 1, 1};
    for (int k = 0; k < 4; k++) {
        J.old_dirty[k] = max_len;
        if (!fixed || !planes4[k]) continue;
        auto it = h->plane_meta.find(planes4[k]);
        if (it != h->plane_meta.end() && it->second.rows == n && it->second.width == max_len && it->second.elt == elts4[k]) J.old_dirty[k] = it->second.dirty_cols;
    }

    // every device writes its own rows of the result; the documents are balanced by bytes
    const int G = (int)h->devs.size();
    const std::vector<int64_t> dcut = shard_rows(G, n, [&](int64_t r) { return text_off[r] + (has_pair ? pair_off[r] : 0) + 64 * r; });
    if (rows) {
        std::vector<WindowPart> parts((size_t)G);
        run_parts(h, J, dcut, parts, [&](DeviceCtx* d, const std::vector<int64_t>& cuts, WindowPart* pt) { windows_chunks(h, d, J, 0, nullptr, cuts, pt); });
        for (auto& pt : parts)
            if (pt.status.rc) { free_nolock(); return pt.status.report(h); }
        for (auto& pt : parts) { out->real_tokens += pt.tokens; out->d2h_bytes += pt.d2h_bytes; }
        if (J.want_tt) for (int64_t r = 0; r < n; r++) out->tt_len[r] = max_len;
        return GENZTOK_OK;
    }
    std::vector<EncodePart> parts((size_t)G);
    run_parts(h, J, dcut, parts, [&](DeviceCtx* d, const std::vector<int64_t>& cuts, EncodePart* pt) {
        if (fixed) encode_fixed_chunks(h, d, J, cuts, pt); else encode_ragged_chunks(h, d, J, cuts, pt);
    });
    for (auto& pt : parts)
        if (pt.status.rc) { free_nolock(); return pt.status.report(h); }
    out->real_tokens = 0;
    out->d2h_bytes = 0;
    for (auto& pt : parts) { out->real_tokens += pt.tokens; out->d2h_bytes += pt.d2h_bytes; }
    if (fixed) {
        int32_t extent = 1;
        for (auto& pt : parts) extent = std::max(extent, pt.extent);
        for (int k = 0; k < 4; k++)
            if (planes4[k]) h->plane_meta[planes4[k]] = genztok::PlaneMeta{n, max_len, std::min<int32_t>(max_len, (extent + 31) & ~31), elts4[k], 0};   // (a lower bound of what was copied is enough: the columns behind it hold padding either way)
        if (J.want_tt) for (int64_t r = 0; r < n; r++) out->tt_len[r] = max_len;
    } else {
        // stitch the parts: shift every part's row offsets by what came before it, concatenate the flat planes
        int64_t base = 0, sbase = 0;
        size_t ntot = 0, stot = 0;
        int holders = 0;
        for (auto& pt : parts) { ntot += pt.ids.size(); stot += pt.spans.size(); holders += (pt.ids.size() || pt.spans.size()) ? 1 : 0; }
        if (holders == 1) {
            // one device holds the whole result: its pinned buffers become the caller's (no second copy); they return to the pool on free
            for (auto& pt : parts) {
                if (!(pt.ids.size() || pt.spans.size())) continue;
                auto adopt = [&](auto& v) { auto* q = v.p; if (q) { ob->pinned.push_back({q, v.cap_bytes}); v.p = nullptr; v.cap_bytes = 0; v.n = 0; } return q; };
                out->total = pt.total;
                out->input_ids = adopt(pt.ids); out->attention_mask = adopt(pt.mask);
                if (has_pair) { out->token_type_ids = adopt(pt.tt); out->sequence_id = adopt(pt.seq); }
                if (J.want_spans) out->spans = adopt(pt.spans);
                if (J.want_offs) out->offsets = adopt(pt.tok_offs);
            }
            auto some = [&](size_t bytes) { void* q = malloc(bytes); ob->mallocs.push_back(q); return q; };   // (empty planes still get an address)
            if (!out->input_ids) out->input_ids = (int32_t*)some(16);
            if (!out->attention_mask) out->attention_mask = (uint8_t*)some(16);
            if (has_pair && !out->token_type_ids) out->token_type_ids = (int8_t*)some(16);
            if (has_pair && !out->sequence_id) out->sequence_id = (int8_t*)some(16);
            if (J.want_spans && !out->spans) out->spans = (int32_t*)some(16);
            if (J.want_offs && !out->offsets) out->offsets = (int32_t*)some(16);
            return fixed_layout ? present_fixed() : GENZTOK_OK;
        }
        int32_t* ids = (int32_t*)malloc(std::max<size_t>(ntot * 4, 16)); ob->mallocs.push_back(ids);
        uint8_t* mask = (uint8_t*)malloc(std::max<size_t>(ntot, 16)); ob->mallocs.push_back(mask);
        int8_t *tt = nullptr, *seq = nullptr; int32_t* spans = nullptr;
        if (has_pair) { tt = (int8_t*)malloc(std::max<size_t>(ntot, 16)); ob->mallocs.push_back(tt); seq = (int8_t*)malloc(std::max<size_t>(ntot, 16)); ob->mallocs.push_back(seq); }
        if (J.want_spans) { spans = (int32_t*)malloc(std::max<size_t>(stot * 4, 16)); ob->mallocs.push_back(spans); }
        int32_t* toffs = nullptr;
        if (J.want_offs) { toffs = (int32_t*)malloc(std::max<size_t>(ntot * 8, 16)); ob->mallocs.push_back(toffs); }
        for (int g = 0; g < G; g++) {
            EncodePart& pt = parts[(size_t)g];
            const int64_t rb = dcut[(size_t)g], re = dcut[(size_t)g + 1];
            if (base) for (int64_t r = rb + 1; r <= re; r++) out->row_off[r] += base;
            if (J.want_spans && sbase) for (int64_t r = rb + 1; r <= re; r++) out->span_off[r] += sbase;
            if (!pt.ids.empty()) {
                memcpy(ids + base, pt.ids.data(), pt.ids.size() * 4);
                memcpy(mask + base, pt.mask.data(), pt.mask.size());
                if (has_pair) { memcpy(tt + base, pt.tt.data(), pt.tt.size()); memcpy(seq + base, pt.seq.data(), pt.seq.size()); }
                if (J.want_offs) memcpy(toffs + 2 * base, pt.tok_offs.data(), pt.ids.size() * 8);
            }
            if (J.want_spans && !pt.spans.empty()) memcpy(spans + 2 * sbase, pt.spans.data(), pt.spans.size() * 4);
            base += pt.total; sbase += pt.span_total;
        }
        out->total = base;
        out->input_ids = ids; out->attention_mask = mask; out->token_type_ids = tt; out->sequence_id = seq; out->spans = spans;
        out->offsets = toffs;
        if (fixed_layout) return present_fixed();
    }
    return GENZTOK_OK;
}

// The argument checks both BPE-dropout encodes share (include/genztok.h).
int check_dropout_args(genztok_t* h, const char* what, int64_t n, int32_t max_len, uint32_t flags, double p) {
    if (n < 0) return fail(h, GENZTOK_E_INVALID, "%s: n >= 0 needed (got %lld)", what, (long long)n);
    if (!(p >= 0.0 && p <= 1.0)) return fail(h, GENZTOK_E_INVALID, "%s: the dropout probability must be in [0, 1] (got %g)", what, p);
    if (max_len < 4) return fail(h, GENZTOK_E_INVALID, "%s: BPE-dropout needs the fixed layout with max_len >= 4 (got %d)", what, max_len);
    if (flags & ~(uint32_t)(GENZTOK_WANT_TOKEN_TYPE | GENZTOK_WANT_SEQUENCE_ID))
        return fail(h, GENZTOK_E_INVALID, "%s: BPE-dropout takes only GENZTOK_WANT_TOKEN_TYPE and GENZTOK_WANT_SEQUENCE_ID (no offsets, spans or "
                    "truncation strategy; got flags 0x%x)", what, flags);
    return GENZTOK_OK;
}

}  // namespace

extern "C" {

int genztok_encode_dropout(genztok_t* h, const uint8_t* text, const int64_t* text_off, const uint8_t* pair, const int64_t* pair_off, int64_t n,
                           int32_t max_len, uint32_t flags, double p, uint64_t seed, const int64_t* row_keys, genztok_encoded_t* out) {
    if (!h) return GENZTOK_E_INVALID;
    if (!out || !text_off) return fail(h, GENZTOK_E_INVALID, "genztok_encode_dropout: bad arguments");
    const int rc = check_dropout_args(h, "genztok_encode_dropout", n, max_len, flags, p);
    if (rc) return rc;
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    const DropSpec drop{p, seed, row_keys};
    return encode_host(h, text, text_off, pair, pair_off, n, max_len, 1, 1, flags, 0, &drop, out);
}

int genztok_encode_dropout_device(genztok_t* h, int dev, const uint8_t* d_text, const int64_t* d_text_off, int64_t text_bytes, const uint8_t* d_pair,
                                  const int64_t* d_pair_off, int64_t pair_bytes, int64_t n, int32_t max_len, uint32_t flags, double p, uint64_t seed,
                                  const int64_t* d_row_keys, const genztok_dev_planes_t* planes, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    int rc = check_dropout_args(h, "genztok_encode_dropout_device", n, max_len, flags, p);
    if (rc) return rc;
    if (!d_text_off || (text_bytes > 0 && !d_text) || (d_pair_off && pair_bytes > 0 && !d_pair) || !planes || !planes->input_ids ||
        !planes->attention_mask || !planes->row_len)
        return fail(h, GENZTOK_E_INVALID, "genztok_encode_dropout_device: bad arguments (input_ids, attention_mask and row_len are required)");
    if (((uintptr_t)d_text & 15) || ((uintptr_t)d_pair & 15)) return fail(h, GENZTOK_E_INVALID, "device text buffers must be 16-byte aligned");
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d (handle has %d)", dev, (int)h->devs.size());
    const bool has_pair = d_pair_off != nullptr;
    const int64_t bytes = text_bytes + (has_pair ? pair_bytes : 0);
    if (bytes > h->max_chunk_bytes) return fail(h, GENZTOK_E_LIMIT, "chunk of %lld bytes exceeds max_chunk_bytes=%lld", (long long)bytes, (long long)h->max_chunk_bytes);
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    rc = stream_enter(h, d, st);
    if (rc) return rc;
    if (!d->cache_ready) { rc = ensure_cache(h, d, st, 0); if (rc) return rc; }   // (the counters; the word cache itself is not used)
    if (n > 0) {
        const Side a{d_text, d_text_off, text_bytes}, b{d_pair, d_pair_off, pair_bytes};
        rc = dropout_layout(h, d, st, a, has_pair ? &b : nullptr, n, max_len, p, seed, d_row_keys, 0);
        if (!rc) rc = windows_write(h, d, st, has_pair, n, max_len, 0, STREAMS_CAPPED, flags, nullptr, n, *planes, nullptr, nullptr, 0);
        if (rc) return rc;
    }
    return stream_leave(h, d, st);
}

}  // extern "C"

namespace {

int check_window_args(genztok_t* h, int32_t max_len, int32_t stride, uint32_t flags) {
    if (max_len < 3) return fail(h, GENZTOK_E_INVALID, "windows need max_len >= 3 (got %d)", max_len);
    if (stride < 0 || stride >= max_len - 2) return fail(h, GENZTOK_E_INVALID, "windows need 0 <= stride < max_len - 2 (got stride=%d, max_len=%d)", stride, max_len);
    if (flags & GENZTOK_WANT_SPANS) return fail(h, GENZTOK_E_INVALID, "spans are not available for windows");
    return GENZTOK_OK;
}

}  // namespace

extern "C" {

int genztok_encode_windows(genztok_t* h, const uint8_t* text, const int64_t* text_off, const uint8_t* pair, const int64_t* pair_off, int64_t n,
                           int32_t max_len, int32_t stride, uint32_t flags, genztok_windows_t* out) {
    if (!h) return GENZTOK_E_INVALID;
    if (!out || n < 0 || !text_off) return fail(h, GENZTOK_E_INVALID, "genztok_encode_windows: bad arguments");
    int rc = check_window_args(h, max_len, stride, flags);
    if (rc) return rc;
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    memset(out, 0, sizeof *out);
    std::lock_guard<std::mutex> lk(h->mu);
    EncodeJob J = make_job(text, text_off, pair, pair_off, max_len, flags);
    const bool has_pair = J.has_pair;
    OutBlock* ob = new OutBlock();
    auto bail = [&](int code) { discard_block(h, ob); memset(out, 0, sizeof *out); return code; };
    // every result buffer leaves the pool to hold windows: what plane_meta knew of it no longer holds
    auto take = [&](auto* p) { if (p) h->plane_meta.erase(p); return p; };
    int64_t* win_off = take(out_alloc<int64_t>(h, ob, (size_t)n + 1));
    if (!win_off) return bail(fail(h, GENZTOK_E_NOMEM, "pinned host allocation failed"));
    win_off[0] = 0;
    // shard the documents across the devices as genztok_encode does: contiguous ranges balanced by bytes
    const int G = (int)h->devs.size();
    const std::vector<int64_t> dcut = shard_rows(G, n, [&](int64_t r) { return text_off[r] + (has_pair ? pair_off[r] : 0) + 64 * r; });
    std::vector<WindowPart> parts((size_t)G);
    run_parts(h, J, dcut, parts, [&](DeviceCtx* d, const std::vector<int64_t>& cuts, WindowPart* pt) { windows_chunks(h, d, J, stride, win_off, cuts, pt); });
    for (auto& pt : parts)
        if (pt.status.rc) return bail(pt.status.report(h));
    int64_t K = 0;
    for (auto& pt : parts) K += pt.n_win;
    const size_t tot = (size_t)K * (size_t)max_len;
    genztok_encoded_t& E = out->enc;
    E.n = K; E.total = (int64_t)tot; E.width = max_len; E.has_pair = has_pair;
    E.input_ids = take(out_alloc<int32_t>(h, ob, tot));
    E.attention_mask = take(out_alloc<uint8_t>(h, ob, tot));
    E.row_len = take(out_alloc<int32_t>(h, ob, (size_t)K));
    out->win_doc = take(out_alloc<int64_t>(h, ob, (size_t)K));
    out->win_start = take(out_alloc<int32_t>(h, ob, (size_t)K));
    bool ok = E.input_ids && E.attention_mask && E.row_len && out->win_doc && out->win_start;
    if (J.want_tt) { E.token_type_ids = take(out_alloc<int8_t>(h, ob, tot)); E.tt_len = take(out_alloc<int32_t>(h, ob, (size_t)K)); ok = ok && E.token_type_ids && E.tt_len; }
    if (J.want_seq) { E.sequence_id = take(out_alloc<int8_t>(h, ob, tot)); ok = ok && E.sequence_id; }
    if (J.want_offs) { E.offsets = take(out_alloc<int32_t>(h, ob, 2 * tot)); ok = ok && E.offsets; }
    if (has_pair) { E.seq_len = take(out_alloc<int32_t>(h, ob, (size_t)K)); E.row_status = take(out_alloc<uint8_t>(h, ob, (size_t)K)); ok = ok && E.seq_len && E.row_status; }
    if (!ok) return bail(fail(h, GENZTOK_E_NOMEM, "pinned host allocation failed"));
    // stitch the parts in document order; their window offsets are shifted by the windows before them
    int64_t base = 0;
    for (int g = 0; g < G; g++) {
        WindowPart& pt = parts[(size_t)g];
        if (base) for (int64_t r = dcut[(size_t)g] + 1; r <= dcut[(size_t)g + 1]; r++) win_off[r] += base;
        const size_t k = (size_t)pt.n_win, o = (size_t)base, w = (size_t)max_len;
        if (k) {
            memcpy(E.input_ids + o * w, pt.ids.data(), k * w * 4);
            memcpy(E.attention_mask + o * w, pt.mask.data(), k * w);
            memcpy(E.row_len + o, pt.row_len.data(), k * 4);
            memcpy(out->win_doc + o, pt.doc.data(), k * 8);
            memcpy(out->win_start + o, pt.start.data(), k * 4);
            if (J.want_tt) memcpy(E.token_type_ids + o * w, pt.tt.data(), k * w);
            if (J.want_seq) memcpy(E.sequence_id + o * w, pt.seq.data(), k * w);
            if (J.want_offs) memcpy(E.offsets + 2 * o * w, pt.tok_offs.data(), k * w * 8);
            if (has_pair) { memcpy(E.seq_len + o, pt.seq_len.data(), k * 4); memcpy(E.row_status + o, pt.row_status.data(), k); }
        }
        base += pt.n_win;
        E.real_tokens += pt.tokens; E.d2h_bytes += pt.d2h_bytes;
    }
    if (J.want_tt) for (int64_t r = 0; r < K; r++) E.tt_len[r] = max_len;
    E._owner = ob;
    out->n_docs = n;
    out->win_off = win_off;
    return GENZTOK_OK;
}

void genztok_free_windows(genztok_t* h, genztok_windows_t* out) {
    if (!out) return;
    genztok_free_encoded(h, &out->enc);                              // (the maps belong to the same block)
    memset(out, 0, sizeof *out);
}

int genztok_encode_windows_device(genztok_t* h, int dev, const uint8_t* d_text, const int64_t* d_text_off, int64_t text_bytes, const uint8_t* d_pair,
                                  const int64_t* d_pair_off, int64_t pair_bytes, int64_t n, int32_t max_len, int32_t stride, uint32_t flags,
                                  int64_t* d_win_off, const genztok_dev_planes_t* planes, int64_t* d_win_doc, int32_t* d_win_start, int64_t* n_windows,
                                  void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d (handle has %d)", dev, (int)h->devs.size());
    if (n < 0 || !d_text_off || !d_win_off || (text_bytes > 0 && !d_text) || (planes == nullptr && !n_windows))
        return fail(h, GENZTOK_E_INVALID, "genztok_encode_windows_device: bad arguments");
    int rc = check_window_args(h, max_len, stride, flags);
    if (rc) return rc;
    if (((uintptr_t)d_text & 15) || ((uintptr_t)d_pair & 15)) return fail(h, GENZTOK_E_INVALID, "device text buffers must be 16-byte aligned");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    const bool has_pair = d_pair_off != nullptr;
    const int64_t bytes = text_bytes + (has_pair ? pair_bytes : 0);
    if (bytes > h->max_chunk_bytes) return fail(h, GENZTOK_E_LIMIT, "chunk of %lld bytes exceeds max_chunk_bytes=%lld", (long long)bytes, (long long)h->max_chunk_bytes);
    DeviceCtx::WinState& S = d->win;
    const bool offs = (flags & GENZTOK_WANT_OFFSETS) != 0;
    const bool same = S.n_win >= 0 && S.sig.a == d_text && S.sig.a_off == d_text_off && S.sig.b == d_pair && S.sig.b_off == d_pair_off &&
                      S.sig.win_off == d_win_off && S.sig.n == n && S.sig.a_bytes == text_bytes && S.sig.b_bytes == (has_pair ? pair_bytes : 0) &&
                      S.sig.W == max_len && S.sig.s == stride && S.sig.offs == offs;
    rc = stream_enter(h, d, st);
    if (rc) return rc;
    if (!planes || !same) {
        int64_t K = 0;
        if (n == 0) CU(cudaMemsetAsync(d_win_off, 0, 8, st));
        else {
            rc = ensure_cache(h, d, st, bytes + 32);
            if (rc) return rc;
            Side a{d_text, d_text_off, text_bytes}, b{d_pair, d_pair_off, pair_bytes};
            rc = windows_layout(h, d, st, a, has_pair ? &b : nullptr, n, max_len, stride, 0, offs, d_win_off, &K);
            if (rc) return rc;
        }
        S.n_win = K;
        S.sig.a = d_text; S.sig.a_off = d_text_off; S.sig.b = d_pair; S.sig.b_off = d_pair_off; S.sig.win_off = d_win_off;
        S.sig.n = n; S.sig.a_bytes = text_bytes; S.sig.b_bytes = has_pair ? pair_bytes : 0; S.sig.W = max_len; S.sig.s = stride; S.sig.offs = offs;
    }
    if (n_windows) *n_windows = S.n_win;
    if (planes) {
        if (S.n_win > 0 && (!planes->input_ids || !planes->attention_mask || !planes->row_len || !d_win_doc || !d_win_start))
            return fail(h, GENZTOK_E_INVALID, "genztok_encode_windows_device: step 2 needs input_ids, attention_mask, row_len and the two maps");
        if (S.n_win > 0 && offs && !planes->offsets) return fail(h, GENZTOK_E_INVALID, "genztok_encode_windows_device: GENZTOK_WANT_OFFSETS needs planes->offsets");
        rc = windows_write(h, d, st, has_pair, n, max_len, stride, 0, flags, d_win_off, S.n_win, *planes, d_win_doc, d_win_start, 0);
        if (rc) return rc;
    }
    return stream_leave(h, d, st);
}

}  // extern "C"

namespace {

// Both passes of the decode on one device; the caller holds h->mu (or owns the device context, as the workers of genztok_decode do).
// capacity < 0: the two-step protocol of genztok_decode_device (d_bytes == NULL: sizes; else: the text of the same batch).
// capacity >= 0: both steps at once into d_bytes[capacity] without a host read in between (genztok_decode_device_into).
int decode_on_device_impl(genztok_t* h, DeviceCtx* d, const int32_t* d_ids, const int64_t* d_ids_off, int64_t n, int32_t width, int64_t* d_out_off,
                          uint8_t* d_bytes, int64_t* total_bytes, cudaStream_t st, int64_t capacity = -1);
int decode_on_device(genztok_t* h, DeviceCtx* d, const int32_t* d_ids, const int64_t* d_ids_off, int64_t n, int32_t width, int64_t* d_out_off,
                     uint8_t* d_bytes, int64_t* total_bytes, void* stream, int64_t capacity = -1) {
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    int rc = stream_enter(h, d, st);
    if (rc) return rc;
    rc = decode_on_device_impl(h, d, d_ids, d_ids_off, n, width, d_out_off, d_bytes, total_bytes, st, capacity);
    if (rc) return rc;
    return stream_leave(h, d, st);
}
int decode_on_device_impl(genztok_t* h, DeviceCtx* d, const int32_t* d_ids, const int64_t* d_ids_off, int64_t n, int32_t width, int64_t* d_out_off,
                          uint8_t* d_bytes, int64_t* total_bytes, cudaStream_t st, int64_t capacity) {
    const bool into = capacity >= 0 && d_bytes != nullptr;
    if (capacity >= 0 && !into) { d_bytes = nullptr; }              // nowhere to write: sizes only
    DecArgs A{d_ids, d_ids_off, width, n, nullptr, d_out_off, d_bytes, nullptr, nullptr, nullptr, into ? (long long)std::max<int64_t>(capacity, 1) : 0ll, 0, (int32_t)h->decode_wide_max};
    // fixed-width rows of whole 16-byte vectors whose byte counts fit 32 bits: a warp per 32 rows instead of a warp per row
    const bool fixed = !d_ids_off && width >= 4 && width % 4 == 0 && (reinterpret_cast<uintptr_t>(d_ids) & 15) == 0 &&
                       (int64_t)width * std::max<int64_t>(1, h->H.max_form) < (1ll << 31) && h->no_fixed_decode == 0;
    // one wave of resident blocks (4 per SM by the kernels' launch bounds, 5 for k_decode_write_fixed), rows or tiles of 32 rows by grid stride
    const unsigned grid_len = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 7) / 8, (int64_t)d->sm_count * 4));
    const unsigned grid_write = fixed ? (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 7) / 8, (int64_t)d->sm_count * 5)) : grid_len;
    CU(d->dec_lead.ensure((size_t)std::max<int64_t>(n, 1) * sizeof(DecLead)));
    A.lead = d->dec_lead.as<DecLead>();
    auto same_batch = [&](int by_id_) { return d->dec_sig.ids == (const void*)d_ids && d->dec_sig.ids_off == (const void*)d_ids_off && d->dec_sig.out_off == (const void*)d_out_off &&
                                               d->dec_sig.n == n && d->dec_sig.width == width && d->dec_sig.by_id == by_id_; };
    // Ragged rows: one thread per id (k_dectok_*).  The host needs the number of ids for that: one small read of the offsets.
    const bool by_id = d_ids_off && n > 0 && h->no_token_decode == 0;
    auto length_pass_by_id = [&]() -> int {
        int64_t ends[2] = {0, 0};
        CU(cudaMemcpyAsync(&ends[0], d_ids_off, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(&ends[1], d_ids_off + n, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        const int64_t N = ends[1] - ends[0];
        if (N < 0) return fail(h, GENZTOK_E_INVALID, "genztok_decode_device: id offsets decrease");
        if (N > (1ll << 28)) return 1;                              // too many ids for the per-id work arrays: warp per row
        CU(d->tok_flag.ensure((size_t)N + 16)); CU(d->tok_len.ensure((size_t)(N + 1) * 8)); CU(d->tok_pos.ensure((size_t)(N + 2) * 8));
        DecTokArgs K{d_ids, d_ids_off, n, ends[0], N, d->tok_flag.as<uint8_t>(), d->tok_len.as<int64_t>(), d->tok_pos.as<int64_t>(), d_out_off, nullptr, 0};
        CU(cudaMemsetAsync(K.flag, 0, (size_t)N + 16, st));
        { LaunchScope ls(h, d, "k_dectok_flags"); k_dectok_flags<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(K); }
        if (N > 0) { LaunchScope ls(h, d, "k_dectok_len"); k_dectok_len<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(d->T, K); }
        { int rc = launch_scan(h, d, st, K.len, d->tok_pos.as<int64_t>(), N); if (rc) return rc; }
        { LaunchScope ls(h, d, "k_dectok_rowoff"); k_dectok_rowoff<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(K); }
        CU(cudaGetLastError());
        d->tok_base = ends[0]; d->tok_n = N;
        d->dec_sig.ids = d_ids; d->dec_sig.ids_off = d_ids_off; d->dec_sig.out_off = d_out_off; d->dec_sig.n = n; d->dec_sig.width = width; d->dec_sig.by_id = 1;
        return GENZTOK_OK;
    };
    if (by_id) {
        int rc = GENZTOK_OK;
        if (!d_bytes || into || !same_batch(1) || d->tok_n < 0) {
            rc = length_pass_by_id();
            if (rc < 0) return rc;
        }
        if (rc == GENZTOK_OK) {
            if (!d_bytes) {
                if (total_bytes) {
                    CU(cudaMemcpyAsync(total_bytes, d_out_off + n, 8, cudaMemcpyDeviceToHost, st));
                    CU(cudaStreamSynchronize(st));
                }
                return GENZTOK_OK;
            }
            DecTokArgs K{d_ids, d_ids_off, n, d->tok_base, d->tok_n, d->tok_flag.as<uint8_t>(), d->tok_len.as<int64_t>(), d->tok_pos.as<int64_t>(), d_out_off, d_bytes, A.capacity};
            if (K.n_ids > 0) { LaunchScope ls(h, d, "k_dectok_write"); k_dectok_write<<<(unsigned)((K.n_ids + 255) / 256), 256, 0, st>>>(d->T, K); }
            CU(cudaGetLastError());
            if (into && total_bytes) {
                CU(cudaMemcpyAsync(total_bytes, d_out_off + n, 8, cudaMemcpyDeviceToHost, st));
                CU(cudaStreamSynchronize(st));
            }
            return GENZTOK_OK;
        }
        d->tok_n = -1;                                              // rc == 1: fall through to the warp-per-row kernels
    } else d->tok_n = -1;
    auto length_pass = [&]() -> int {
        CU(d->out_len.ensure((size_t)std::max<int64_t>(n, 1) * 8));
        A.out_len = d->out_len.as<int64_t>();
        d->dec_avg_lead = -1;
        if (fixed) {
            CU(d->dec_stat.ensure(32));
            CU(cudaMemsetAsync(d->dec_stat.p, 0, 16, st));
            A.lead_sum = d->dec_stat.as<unsigned long long>();
            A.tile_ctr = d->dec_stat.as<unsigned long long>() + 1;
        }
        if (n > 0 && fixed) {
            const unsigned grid_fixed = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)d->sm_count * DEC_LEN_MINB));
            LaunchScope ls(h, d, "k_decode_len_fixed");
            if (width <= 128) k_decode_len_fixed<1><<<grid_fixed, 256, 0, st>>>(d->T, A);
            else if (width <= 256) k_decode_len_fixed<2><<<grid_fixed, 256, 0, st>>>(d->T, A);
            else k_decode_len_fixed<0><<<grid_fixed, 256, 0, st>>>(d->T, A);
        }
        else if (n > 0) { LaunchScope ls(h, d, "k_decode_len"); k_decode_len<<<grid_len, 256, 0, st>>>(d->T, A); }
        d->dec_sig.ids = d_ids; d->dec_sig.ids_off = d_ids_off; d->dec_sig.out_off = d_out_off; d->dec_sig.n = n; d->dec_sig.width = width; d->dec_sig.by_id = 0;
        return GENZTOK_OK;
    };
    if (!d_bytes) {
        { int rc = length_pass(); if (rc) return rc; }
        { int rc = launch_scan(h, d, st, d->out_len.as<int64_t>(), d_out_off, n); if (rc) return rc; }
        if (total_bytes) {
            unsigned long long lead_sum = 0;
            CU(cudaMemcpyAsync(total_bytes, d_out_off + n, 8, cudaMemcpyDeviceToHost, st));
            if (fixed) CU(cudaMemcpyAsync(&lead_sum, d->dec_stat.p, 8, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            if (fixed && n > 0) d->dec_avg_lead = (double)lead_sum / (double)n;
        }
        return GENZTOK_OK;
    }
    // the write pass reads what the length pass of the same batch left in dec_lead; after another batch's length pass it is redone
    if (into) {
        { int rc = length_pass(); if (rc) return rc; }
        { int rc = launch_scan(h, d, st, d->out_len.as<int64_t>(), d_out_off, n); if (rc) return rc; }
    } else if (!same_batch(0)) { int rc = length_pass(); if (rc) return rc; }
    // Three write kernels for fixed-width rows: a lane per junction of two rows assembles short leads (single sentences, ~10 pieces in
    // front of the pad run) in 256 bytes, longer ones in 512; the whole warp gathers the longest 32 pieces at a time.  The length pass
    // counted the pieces.  Without a host read in between (into) all three are launched and the batch's count picks one on the device.
    int by_lanes = h->decode_write == 2 ? 1 : h->decode_write == 3 ? 2 : h->decode_write == 1 ? 3 : 0;
    if (by_lanes == 0 && !into) by_lanes = d->dec_avg_lead < 0 ? 3 : dec_pick((unsigned long long)(d->dec_avg_lead * (double)n + 0.5), n, (int)h->decode_wide_max);
    A.pick = (into && fixed && by_lanes == 0) ? 1 : 0;
    auto launch_junctions = [&](auto kern, int stride, int warps) -> int {
        const size_t smem = (size_t)warps * (32 * (size_t)stride + 16);
        CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ = 1;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, warps * 32, smem));
        const int64_t per_block = 32 * warps;
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 1 + per_block - 1) / per_block, (int64_t)d->sm_count * std::max(occ, 1)));   // n + 1 junctions
        LaunchScope ls(h, d, "k_decode_write_fixed");
        kern<<<grid, warps * 32, smem, st>>>(d->T, A);
        return GENZTOK_OK;
    };
    if (n > 0 && fixed) {
        CU(d->dec_stat.ensure(32));
        CU(cudaMemsetAsync(d->dec_stat.as<unsigned long long>() + 2, 0, 8, st));
        A.tile_ctr = d->dec_stat.as<unsigned long long>() + 2;          // (one counter: only the kernel that writes takes tiles)
        if (A.pick || by_lanes == 1) { int rc = launch_junctions(k_decode_write_fixed<256, 8, 3>, 256, 8); if (rc) return rc; }
        if ((A.pick && h->decode_wide_max > 14) || by_lanes == 2) { int rc = launch_junctions(k_decode_write_fixed<512, 4, 3>, 512, 4); if (rc) return rc; }
        if (A.pick || by_lanes == 3) {
            LaunchScope ls(h, d, "k_decode_write_fixed");
            k_decode_write_fixed_coop<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)d->sm_count * 5)), 256, 0, st>>>(d->T, A);
        }
    }
    else if (n > 0) { LaunchScope ls(h, d, "k_decode_write"); k_decode_write<<<grid_write, 256, 0, st>>>(d->T, A); }
    if (into && total_bytes) {
        CU(cudaMemcpyAsync(total_bytes, d_out_off + n, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

}  // namespace

extern "C" {

int genztok_decode_device(genztok_t* h, int dev, const int32_t* d_ids, const int64_t* d_ids_off, int64_t n, int32_t width, int64_t* d_out_off,
                          uint8_t* d_bytes, int64_t* total_bytes, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    if (n < 0 || !d_out_off || (!d_ids_off && width < 0)) return fail(h, GENZTOK_E_INVALID, "genztok_decode_device: bad arguments");
    std::lock_guard<std::mutex> lk(h->mu);
    return decode_on_device(h, h->devs[(size_t)dev], d_ids, d_ids_off, n, width, d_out_off, d_bytes, total_bytes, stream);
}

int genztok_decode_device_into(genztok_t* h, int dev, const int32_t* d_ids, const int64_t* d_ids_off, int64_t n, int32_t width, int64_t* d_out_off,
                               uint8_t* d_bytes, int64_t capacity, int64_t* total_bytes, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    if (n < 0 || !d_out_off || capacity < 0 || (!d_ids_off && width < 0)) return fail(h, GENZTOK_E_INVALID, "genztok_decode_device_into: bad arguments");
    std::lock_guard<std::mutex> lk(h->mu);
    return decode_on_device(h, h->devs[(size_t)dev], d_ids, d_ids_off, n, width, d_out_off, d_bytes, total_bytes, stream, capacity);
}

void genztok_free_text(genztok_t* h, genztok_text_t* out) { free_result(h, out); }

}  // extern "C"

namespace {

struct DecodePart { PartStatus status; std::vector<uint8_t> bytes; std::vector<int64_t> off; };   // off: row ends relative to the part's start

// Rows [r0, r1) on one device, in chunks of chunk_rows: ids up, both passes, text and offsets down.
void decode_rows_on_device(genztok_t* h, DeviceCtx* d, const int32_t* ids, const int64_t* ids_off, int32_t width, int64_t r0, int64_t r1, DecodePart* part) {
    cudaStream_t st = d->stream;
    CUF(cudaSetDevice(d->device));
    const int64_t rows_per_chunk = std::max<int64_t>(1, h->chunk_rows);
    part->off.reserve((size_t)(r1 - r0));
    int64_t total_all = 0;
    std::vector<int64_t> offs;
    for (int64_t c0 = r0; c0 < r1; c0 += rows_per_chunk) {
        const int64_t c1 = std::min(r1, c0 + rows_per_chunk), m = c1 - c0;
        const int64_t i0 = ids_off ? ids_off[c0] : c0 * width, i1 = ids_off ? ids_off[c1] : c1 * width, ni = i1 - i0;
        cudaError_t e;
        if ((e = d->ids.ensure((size_t)ni * 4 + 16)) != cudaSuccess || (e = d->row_off.ensure((size_t)(m + 1) * 8)) != cudaSuccess ||
            (e = d->toff.ensure((size_t)(m + 1) * 8)) != cudaSuccess) PFAIL(GENZTOK_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(e))
        if (ni) CUF(cudaMemcpyAsync(d->ids.p, ids + i0, (size_t)ni * 4, cudaMemcpyHostToDevice, st));
        const int64_t* d_ioff = nullptr;
        if (ids_off) { CUF(cudaMemcpyAsync(d->toff.p, ids_off + c0, (size_t)(m + 1) * 8, cudaMemcpyHostToDevice, st)); d_ioff = d->toff.as<int64_t>(); }
        int64_t total = 0;
        FAIL_RC(decode_on_device(h, d, d->ids.as<int32_t>() - (ids_off ? i0 : 0), d_ioff, m, width, d->row_off.as<int64_t>(), nullptr, &total, st));
        if ((e = d->text.ensure((size_t)total + 16)) != cudaSuccess) PFAIL(GENZTOK_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(e))
        FAIL_RC(decode_on_device(h, d, d->ids.as<int32_t>() - (ids_off ? i0 : 0), d_ioff, m, width, d->row_off.as<int64_t>(), d->text.as<uint8_t>(), nullptr, st));
        offs.resize((size_t)m + 1);
        const size_t old = part->bytes.size();
        part->bytes.resize(old + (size_t)total);
        if (total) CUF(cudaMemcpyAsync(part->bytes.data() + old, d->text.p, (size_t)total, cudaMemcpyDeviceToHost, st));
        CUF(cudaMemcpyAsync(offs.data(), d->row_off.p, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) PFAIL(GENZTOK_E_CUDA, "decode: %s", cudaGetErrorString(e))
        for (int64_t i = 1; i <= m; i++) part->off.push_back(total_all + offs[(size_t)i]);
        total_all += total;
    }
}

}  // namespace

extern "C" {

int genztok_decode(genztok_t* h, const int32_t* ids, const int64_t* ids_off, int64_t n, int32_t width, genztok_text_t* out) {
    if (!h) return GENZTOK_E_INVALID;
    if (!out || n < 0 || (!ids_off && width < 0)) return fail(h, GENZTOK_E_INVALID, "genztok_decode: bad arguments");
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    memset(out, 0, sizeof *out);
    std::lock_guard<std::mutex> lk(h->mu);
    OutBlock* ob = new OutBlock();
    int64_t* off = out_alloc<int64_t>(h, ob, (size_t)n + 1);
    if (!off) { delete ob; return fail(h, GENZTOK_E_NOMEM, "pinned host allocation failed"); }
    off[0] = 0;
    // the rows are balanced by ids; the parts' texts are concatenated and their offsets shifted
    const int G = (int)h->devs.size();
    const std::vector<int64_t> dcut = shard_rows(G, n, [&](int64_t r) { return (ids_off ? ids_off[r] - ids_off[0] : r * (int64_t)width) + 16 * r; });
    std::vector<DecodePart> parts((size_t)G);
    run_shards(dcut, [&](int g) { decode_rows_on_device(h, h->devs[(size_t)g], ids, ids_off, width, dcut[(size_t)g], dcut[(size_t)g + 1], &parts[(size_t)g]); });
    for (auto& pt : parts)
        if (pt.status.rc) { discard_block(h, ob); return pt.status.report(h); }
    size_t total_all = 0;
    for (auto& pt : parts) total_all += pt.bytes.size();
    uint8_t* bytes = (uint8_t*)malloc(std::max<size_t>(total_all, 16));
    ob->mallocs.push_back(bytes);
    int64_t base = 0, row = 0;
    for (auto& pt : parts) {
        if (!pt.bytes.empty()) memcpy(bytes + base, pt.bytes.data(), pt.bytes.size());
        for (int64_t v : pt.off) off[++row] = base + v;
        base += (int64_t)pt.bytes.size();
    }
    out->n = n; out->total = (int64_t)total_all; out->bytes = bytes; out->off = off; out->_owner = ob;
    return GENZTOK_OK;
}

// ---- preprocess.py normalisers ------------------------------------------------------------------------------
int genztok_preprocess(genztok_t* h, int op, const uint8_t* text, const int64_t* text_off, int64_t n, genztok_text_t* out) {
    if (!h) return GENZTOK_E_INVALID;
    if (!out || n < 0 || !text_off || op < 0 || op > 4) return fail(h, GENZTOK_E_INVALID, "genztok_preprocess: bad arguments");
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    memset(out, 0, sizeof *out);
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[0];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = d->stream;
    LaunchScope::cur_stream = st;
    int rc = stream_enter(h, d, st);                                 // (the text, offset and length buffers are the encode's too)
    if (rc) return rc;
    OutBlock* ob = new OutBlock();
    int64_t* off = out_alloc<int64_t>(h, ob, (size_t)n + 1);
    if (!off) { delete ob; return fail(h, GENZTOK_E_NOMEM, "pinned host allocation failed"); }
    off[0] = 0;
    std::vector<uint8_t> acc;
    int64_t total_all = 0;
    auto bail = [&](int code) { discard_block(h, ob); return code; };
    int64_t r0 = 0;
    while (r0 < n) {
        int64_t r1 = std::min<int64_t>(n, r0 + h->chunk_rows);
        while (r1 > r0 + 1 && text_off[r1] - text_off[r0] > h->max_chunk_bytes) r1 = r0 + (r1 - r0) / 2;
        const int64_t m = r1 - r0, b0 = text_off[r0], nb = text_off[r1] - b0;
        cudaError_t e;
        if ((e = d->text.ensure((size_t)nb + 64)) != cudaSuccess || (e = d->toff.ensure((size_t)(m + 1) * 8)) != cudaSuccess ||
            (e = d->out_len.ensure((size_t)m * 8)) != cudaSuccess || (e = d->row_off.ensure((size_t)(m + 1) * 8)) != cudaSuccess)
            return bail(fail(h, GENZTOK_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(e)));
        if (nb) cudaMemcpyAsync(d->text.p, text + b0, (size_t)nb, cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d->toff.p, text_off + r0, (size_t)(m + 1) * 8, cudaMemcpyHostToDevice, st);
        PrepArgs A{d->text.as<uint8_t>() - b0, d->toff.as<int64_t>(), m, op, d->out_len.as<int64_t>(), d->row_off.as<int64_t>(), nullptr};
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((m + 7) / 8, (int64_t)d->sm_count * 8));
        { LaunchScope ls(h, d, "k_prep_len"); k_prep<false><<<grid, 256, 0, st>>>(A); }
        rc = launch_scan(h, d, st, d->out_len.as<int64_t>(), d->row_off.as<int64_t>(), m);
        if (rc) return bail(rc);
        int64_t total = 0;
        cudaMemcpyAsync(&total, d->row_off.as<int64_t>() + m, 8, cudaMemcpyDeviceToHost, st);
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return bail(fail(h, GENZTOK_E_CUDA, "preprocess: %s", cudaGetErrorString(e)));
        if ((e = d->prep_out.ensure((size_t)total + 64)) != cudaSuccess) return bail(fail(h, GENZTOK_E_CUDA, "cudaMalloc: %s", cudaGetErrorString(e)));
        A.out = d->prep_out.as<uint8_t>();
        { LaunchScope ls(h, d, "k_prep_write"); k_prep<true><<<grid, 256, 0, st>>>(A); }
        std::vector<int64_t> offs((size_t)m + 1);
        const size_t old = acc.size();
        acc.resize(old + (size_t)total);
        if (total) cudaMemcpyAsync(acc.data() + old, d->prep_out.p, (size_t)total, cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(offs.data(), d->row_off.p, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st);
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return bail(fail(h, GENZTOK_E_CUDA, "preprocess: %s", cudaGetErrorString(e)));
        for (int64_t i = 1; i <= m; i++) off[r0 + i] = total_all + offs[(size_t)i];
        total_all += total;
        r0 = r1;
    }
    rc = stream_leave(h, d, st);
    if (rc) return bail(rc);
    uint8_t* bytes = (uint8_t*)malloc(std::max<size_t>(acc.size(), 16));
    if (!acc.empty()) memcpy(bytes, acc.data(), acc.size());
    ob->mallocs.push_back(bytes);
    out->n = n; out->total = total_all; out->bytes = bytes; out->off = off; out->_owner = ob;
    return GENZTOK_OK;
}

// ---- measurement plumbing: synthetic workload on the device, plane digest, error counter (synth.cuh) ---------------
int genztok_synth_init(genztok_t* h, int dev, const uint8_t* wblob, int64_t wblob_len, const uint32_t* wstart, const uint32_t* wlen, const uint32_t* cdf32,
                       int64_t nw, const uint8_t* eblob, int64_t eblob_len, const uint32_t* estart, const uint32_t* elen, int64_t ne) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    if (!wblob || !wstart || !wlen || !cdf32 || nw < 1 || !eblob || !estart || !elen || ne < 1) return fail(h, GENZTOK_E_INVALID, "genztok_synth_init: bad arguments");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    SynthTables& S = d->synth;
    CU(upload(d, std::vector<uint8_t>(wblob, wblob + wblob_len), &S.wblob));
    CU(upload(d, std::vector<uint32_t>(wstart, wstart + nw), &S.wstart));
    CU(upload(d, std::vector<uint32_t>(wlen, wlen + nw), &S.wlen));
    CU(upload(d, std::vector<uint32_t>(cdf32, cdf32 + nw), &S.cdf32));
    CU(upload(d, std::vector<uint8_t>(eblob, eblob + eblob_len), &S.eblob));
    CU(upload(d, std::vector<uint32_t>(estart, estart + ne), &S.estart));
    CU(upload(d, std::vector<uint32_t>(elen, elen + ne), &S.elen));
    S.nw = (uint32_t)nw; S.ne = (uint32_t)ne;
    d->synth_ready = true;
    return GENZTOK_OK;
}

int genztok_synth_device(genztok_t* h, int dev, uint64_t seed, int64_t doc0, int64_t n, int side, int lo, int hi, uint32_t noise_thr, int64_t* d_off,
                         uint8_t* d_bytes, int64_t* total_bytes, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    if (n < 0 || !d_off || lo < 0 || hi < lo || hi > 4096) return fail(h, GENZTOK_E_INVALID, "genztok_synth_device: bad arguments");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    if (!d->synth_ready) return fail(h, GENZTOK_E_INVALID, "genztok_synth_device: call genztok_synth_init first");
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    SynthArgs A{seed, doc0, n, side, lo, hi, noise_thr, nullptr, d_off, d_bytes};
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)d->sm_count * 16));
    if (!d_bytes) {
        CU(d->synth_len.ensure((size_t)std::max<int64_t>(n, 1) * 8));
        A.len_out = d->synth_len.as<int64_t>();
        if (n > 0) { LaunchScope ls(h, d, "k_synth_len"); k_synth<false><<<grid, 256, 0, st>>>(d->synth, A); }
        int rc = launch_scan(h, d, st, d->synth_len.as<int64_t>(), d_off, n);
        if (rc) return rc;
        if (total_bytes) {
            CU(cudaMemcpyAsync(total_bytes, d_off + n, 8, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
        }
        return GENZTOK_OK;
    }
    if (n > 0) { LaunchScope ls(h, d, "k_synth_write"); k_synth<true><<<grid, 256, 0, st>>>(d->synth, A); }
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

int genztok_digest_device(genztok_t* h, int dev, const int32_t* d_ids, const uint8_t* d_mask, const int8_t* d_tt, int64_t n, int32_t width, int64_t row0,
                          uint64_t* d_acc, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    if (n < 0 || !d_ids || !d_mask || !d_acc || width < 4 || (width & 3)) return fail(h, GENZTOK_E_INVALID, "genztok_digest_device: needs ids, mask and a width that is a multiple of 4");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    DigestArgs A{reinterpret_cast<const uint32_t*>(d_ids), reinterpret_cast<const uint32_t*>(d_mask), reinterpret_cast<const uint32_t*>(d_tt), n, row0, width,
                 reinterpret_cast<unsigned long long*>(d_acc)};
    if (n > 0) { LaunchScope ls(h, d, "k_plane_digest"); k_plane_digest<<<(unsigned)std::min<int64_t>((n + 7) / 8, (int64_t)d->sm_count * 8), 256, 0, st>>>(A); }
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

/* The device pipeline counts inconsistencies (offsets outside the stated text, exhausted work lists) instead of faulting; the
 * host path checks the counter after every call, the asynchronous device path leaves that to the caller: this reads it
 * (synchronises `stream`). */
int genztok_gather_rows(genztok_t* h, int dev, int n_fields, const void* const* d_fields, const int64_t* row_bytes, int64_t n_rows, const int64_t* d_index,
                        int64_t n_index, void* const* d_out, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    if (n_fields < 1 || n_fields > GATHER_MAX_FIELDS || !d_fields || !row_bytes || !d_out || n_rows < 0 || n_index < 0 || (n_index > 0 && !d_index))
        return fail(h, GENZTOK_E_INVALID, "genztok_gather_rows: bad arguments (1..%d fields)", GATHER_MAX_FIELDS);
    GatherArgs A{};
    for (int f = 0; f < n_fields; f++) {
        if (!d_fields[f] || !d_out[f] || row_bytes[f] < 0 || row_bytes[f] >= (1ll << 31)) return fail(h, GENZTOK_E_INVALID, "genztok_gather_rows: field %d", f);
        A.src[f] = static_cast<const uint8_t*>(d_fields[f]); A.dst[f] = static_cast<uint8_t*>(d_out[f]); A.row_bytes[f] = (uint32_t)row_bytes[f];
    }
    A.n_fields = n_fields; A.n_rows = n_rows; A.index = d_index; A.n_index = n_index;
    if (n_index == 0) return GENZTOK_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    {
        LaunchScope ls(h, d, "k_gather_rows");
        k_gather_rows<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((n_index + 7) / 8, (int64_t)d->sm_count * 8)), 256, 0, st>>>(A);
    }
    CU(cudaGetLastError());
    return GENZTOK_OK;
}

// Extractive QA (qa.cuh).  Arguments are checked before the device slot, so that a host-only handle reports them too.  The kernels
// count inconsistent inputs in the word cache's error counter, which is created here when no encode has run on the device yet.
static int qa_enter(genztok_t* h, int dev, void* stream, DeviceCtx** dp, cudaStream_t* stp) {
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d (handle has %d)", dev, (int)h->devs.size());
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    if (!d->cache_ready) { int rc = ensure_cache(h, d, st, 0); if (rc) return rc; }
    *dp = d; *stp = st;
    return stream_enter(h, d, st);
}

int genztok_qa_labels_device(genztok_t* h, int dev, const int32_t* d_offsets, int64_t n_windows, int32_t max_len, int has_pair, const int64_t* d_win_off,
                             int64_t n_docs, const int64_t* d_answers, int unit, const uint8_t* d_text, const int64_t* d_text_off, int64_t text_bytes,
                             int64_t* d_start, int64_t* d_end, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (max_len < 3) return fail(h, GENZTOK_E_INVALID, "genztok_qa_labels_device: max_len >= 3 needed (got %d)", max_len);
    if (unit != GENZTOK_QA_BYTES && unit != GENZTOK_QA_CHARS) return fail(h, GENZTOK_E_INVALID, "genztok_qa_labels_device: unknown unit %d", unit);
    if (n_windows < 0 || n_docs < 0 || !d_win_off || (n_windows > 0 && (!d_offsets || !d_start || !d_end)) || (n_docs > 0 && !d_answers))
        return fail(h, GENZTOK_E_INVALID, "genztok_qa_labels_device: bad arguments");
    if (unit == GENZTOK_QA_CHARS && (!d_text_off || text_bytes < 0 || (text_bytes > 0 && !d_text) || ((uintptr_t)d_text & 15)))
        return fail(h, GENZTOK_E_INVALID, "genztok_qa_labels_device: characters need the text (16-byte aligned) and its offsets");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = nullptr;
    cudaStream_t st = nullptr;
    int rc = qa_enter(h, dev, stream, &d, &st);
    if (rc) return rc;
    QaArgs A{};
    A.om = reinterpret_cast<const int2*>(d_offsets); A.K = n_windows; A.W = max_len; A.pair = has_pair ? 1 : 0;
    A.win_off = d_win_off; A.n = n_docs; A.answers = d_answers; A.start = d_start; A.end = d_end; A.ctr = d->C.ctr;
    if (unit == GENZTOK_QA_CHARS && n_docs > 0) {
        CU(d->qa_ans.ensure((size_t)n_docs * 16));
        A.text = d_text; A.text_off = d_text_off; A.text_bytes = text_bytes; A.char_answers = d_answers; A.byte_answers = d->qa_ans.as<int64_t>();
        A.answers = A.byte_answers;
        LaunchScope ls(h, d, "k_qa_char_to_byte", n_docs * 32 + 8 * (n_docs + 1) + text_bytes);
        k_qa_char_to_byte<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((n_docs + 7) / 8, (int64_t)d->sm_count * 16)), 256, 0, st>>>(A);
    }
    if (n_windows > 0) {
        // om entries read per window: om[0], 32-probe rounds for c1, s and e, and (pairs) the question's columns in rounds of 32
        int64_t rounds = 1;
        for (int64_t r = max_len; r > 32; r = (r + 31) / 32) rounds++;
        const int64_t om_read = 8 + 3 * rounds * 32 * 4 + (has_pair ? 256 : 0);
        LaunchScope ls(h, d, "k_qa_labels", n_windows * (8 + 16 + om_read) + n_docs * 16);
        k_qa_labels<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((n_windows + 7) / 8, (int64_t)d->sm_count * 16)), 256, 0, st>>>(A);
    }
    CU(cudaGetLastError());
    return stream_leave(h, d, st);
}

int genztok_qa_best_spans_device(genztok_t* h, int dev, const float* d_start_logits, const float* d_end_logits, const int32_t* d_offsets, int64_t n_windows,
                                 int32_t max_len, int has_pair, const int64_t* d_win_off, int64_t n_docs, int32_t max_answer_len, float* d_score,
                                 float* d_null_score, int64_t* d_window, int32_t* d_columns, int32_t* d_span, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (max_len < 3) return fail(h, GENZTOK_E_INVALID, "genztok_qa_best_spans_device: max_len >= 3 needed (got %d)", max_len);
    if (max_answer_len < 1) return fail(h, GENZTOK_E_INVALID, "genztok_qa_best_spans_device: max_answer_len >= 1 needed (got %d)", max_answer_len);
    if (n_windows < 0 || n_docs < 0 || !d_win_off || (n_windows > 0 && (!d_start_logits || !d_end_logits || !d_offsets)) ||
        (n_docs > 0 && (!d_score || !d_null_score || !d_window || !d_columns || !d_span)))
        return fail(h, GENZTOK_E_INVALID, "genztok_qa_best_spans_device: bad arguments");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = nullptr;
    cudaStream_t st = nullptr;
    int rc = qa_enter(h, dev, stream, &d, &st);
    if (rc) return rc;
    // a warp stages its window's two logit rows and the two block-maximum arrays: 16 bytes per column
    const size_t per_warp = (size_t)max_len * 16;
    if (per_warp > d->smem_optin) return fail(h, GENZTOK_E_LIMIT, "genztok_qa_best_spans_device: max_len %d needs %zu bytes of shared memory per warp (%zu available)",
                                              max_len, per_warp, d->smem_optin);
    const int wpb = (int)std::max<size_t>(1, std::min<size_t>(8, (48u << 10) / per_warp));
    const size_t smem = per_warp * (size_t)wpb;
    if (smem > (48u << 10)) CU(cudaFuncSetAttribute(k_qa_spans, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    QaArgs A{};
    A.om = reinterpret_cast<const int2*>(d_offsets); A.K = n_windows; A.W = max_len; A.pair = has_pair ? 1 : 0;
    A.win_off = d_win_off; A.n = n_docs; A.S = d_start_logits; A.E = d_end_logits; A.L = std::min(max_answer_len, max_len);
    A.score = d_score; A.null_score = d_null_score; A.window = d_window; A.columns = d_columns; A.span = d_span; A.ctr = d->C.ctr;
    CU(d->qa_win.ensure((size_t)std::max<int64_t>(n_windows, 1) * 16));
    A.w_score = d->qa_win.as<float>(); A.w_null = A.w_score + n_windows;
    A.w_s = reinterpret_cast<int32_t*>(A.w_null + n_windows); A.w_e = A.w_s + n_windows;
    if (n_windows > 0) {
        LaunchScope ls(h, d, "k_qa_spans", n_windows * (int64_t)max_len * (4 + 4 + 8));
        k_qa_spans<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((n_windows + wpb - 1) / wpb, (int64_t)d->sm_count * 32)), 32 * wpb, smem, st>>>(A);
    }
    if (n_docs > 0) {
        LaunchScope ls(h, d, "k_qa_spans_docs", 8 * (n_docs + 1) + n_docs * (4 + 4 + 8 + 8 + 8));
        k_qa_spans_docs<<<(unsigned)std::min<int64_t>((n_docs + 255) / 256, (int64_t)d->sm_count * 8), 256, 0, st>>>(A);
    }
    CU(cudaGetLastError());
    return stream_leave(h, d, st);
}

// MLM masking (mlm.cuh).  Arguments are checked before the device slot, as for the QA calls.
static void mlm_build(genztok_t* h) {
    if (h->mlm_built) return;
    const HostTables& H = h->H;
    h->mlm_cont.assign((size_t)((H.n_ids + 31) / 32), 0u);
    h->mlm_repl.clear();
    for (int64_t id = 0; id < H.n_ids; id++) {
        const int64_t e = H.decoder[(size_t)id];
        if (e < 0) continue;
        const std::string& s = H.enc_keys[(size_t)e];
        if (s.size() >= 2 && s.compare(s.size() - 2, 2, "@@") == 0) h->mlm_cont[(size_t)(id >> 5)] |= 1u << (id & 31);
        if (std::find(H.special_id, H.special_id + 5, (int32_t)id) == H.special_id + 5) h->mlm_repl.push_back((int32_t)id);
    }
    h->mlm_built = true;
}

int genztok_mlm_mask_device(genztok_t* h, int dev, const int32_t* d_ids, int64_t n, int32_t width, const int64_t* d_row_keys, uint64_t seed,
                            double mlm_probability, double mask_replace_prob, double random_replace_prob, int whole_word, int32_t* d_masked_ids,
                            int64_t* d_labels, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    const double p = mlm_probability, a = mask_replace_prob, b = random_replace_prob;
    for (double x : {p, a, b})
        if (!(x >= 0.0 && x <= 1.0))
            return fail(h, GENZTOK_E_INVALID, "genztok_mlm_mask_device: probabilities must be finite and in [0, 1] (got %g, %g, %g)", p, a, b);
    if (a + b > 1.0) return fail(h, GENZTOK_E_INVALID, "genztok_mlm_mask_device: mask_replace_prob + random_replace_prob must be <= 1 (got %g + %g)", a, b);
    if (n < 0 || width < 1) return fail(h, GENZTOK_E_INVALID, "genztok_mlm_mask_device: n >= 0 and width >= 1 needed (got %lld, %d)", (long long)n, width);
    if (n > 0 && (!d_ids || !d_masked_ids || !d_labels)) return fail(h, GENZTOK_E_INVALID, "genztok_mlm_mask_device: ids, masked ids and labels are required");
    if (n > 0 && (const void*)d_masked_ids == (const void*)d_ids)
        return fail(h, GENZTOK_E_INVALID, "genztok_mlm_mask_device: the masked ids must not overwrite the input ids");
    std::lock_guard<std::mutex> lk(h->mu);
    mlm_build(h);
    if (b > 0.0 && h->mlm_repl.empty())
        return fail(h, GENZTOK_E_INVALID, "genztok_mlm_mask_device: random_replace_prob > 0 but the vocab has no id to draw (every id is special)");
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d (handle has %d)", dev, (int)h->devs.size());
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    if (!d->mlm_repl) CU(upload(d, h->mlm_repl, &d->mlm_repl));
    if (!d->mlm_cont) CU(upload(d, h->mlm_cont, &d->mlm_cont));
    int rc = stream_enter(h, d, st);
    if (rc) return rc;
    const double two32 = 4294967296.0;
    MlmArgs A{};
    A.ids = d_ids; A.n = n; A.W = width; A.row_keys = d_row_keys;
    A.s0 = mix64(seed ^ MLM_K);
    A.t_sel = (uint64_t)std::floor(p * two32); A.t_mask = (uint64_t)std::floor(a * two32); A.t_mask_rand = (uint64_t)std::floor((a + b) * two32);
    A.cont = d->mlm_cont; A.repl = d->mlm_repl; A.m = (uint32_t)h->mlm_repl.size(); A.n_ids = d->T.n_ids;
    A.pad = d->T.pad; A.bos = d->T.bos; A.eos = d->T.eos; A.msk = d->T.msk; A.unk = d->T.unk;
    A.out = d_masked_ids; A.labels = d_labels;
    if (n > 0) {
        LaunchScope ls(h, d, whole_word ? "k_mlm_mask_words" : "k_mlm_mask_tokens", n * (int64_t)width * (4 + 4 + 8) + (d_row_keys ? 8 * n : 0));
        const unsigned grid = (unsigned)std::min<int64_t>((n + 7) / 8, (int64_t)d->sm_count * 64);
        if (whole_word) k_mlm_mask<true><<<grid, 256, 0, st>>>(A);
        else k_mlm_mask<false><<<grid, 256, 0, st>>>(A);
    }
    CU(cudaGetLastError());
    return stream_leave(h, d, st);
}

int genztok_check_errors(genztok_t* h, int dev, void* stream, int64_t* n_errors) {
    if (!h || !n_errors) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    *n_errors = 0;
    if (!d->cache_ready) return GENZTOK_OK;
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    unsigned long long nerr = 0;
    CU(cudaMemcpyAsync(&nerr, d->C.ctr + C_ERR, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *n_errors = (int64_t)nerr;
    return nerr ? fail(h, GENZTOK_E_CUDA, "device pipeline reported %llu inconsistencies", nerr) : GENZTOK_OK;
}

// Device form of the normalisers: text and offsets already on the device, the result stays there (so that it can be handed to
// genztok_encode_device on the same stream: normalise -> tokenise without crossing PCIe).  Two steps like genztok_decode_device.
int genztok_preprocess_device(genztok_t* h, int dev, int op, const uint8_t* d_text, const int64_t* d_text_off, int64_t n, int64_t* d_out_off,
                              uint8_t* d_out, int64_t* total_bytes, void* stream) {
    if (!h) return GENZTOK_E_INVALID;
    if (dev < 0 || dev >= (int)h->devs.size()) return fail(h, GENZTOK_E_NODEVICE, "no such device slot %d", dev);
    if (n < 0 || !d_text_off || !d_out_off || op < 0 || op > 4) return fail(h, GENZTOK_E_INVALID, "genztok_preprocess_device: bad arguments");
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[(size_t)dev];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d->stream;
    LaunchScope::cur_stream = st;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 7) / 8, (int64_t)d->sm_count * 8));
    int rc = stream_enter(h, d, st);
    if (rc) return rc;
    if (!d_out) {
        CU(d->out_len.ensure((size_t)std::max<int64_t>(n, 1) * 8));
        PrepArgs A{d_text, d_text_off, n, op, d->out_len.as<int64_t>(), nullptr, nullptr};
        if (n > 0) { LaunchScope ls(h, d, "k_prep_len"); k_prep<false><<<grid, 256, 0, st>>>(A); }
        rc = launch_scan(h, d, st, d->out_len.as<int64_t>(), d_out_off, n);
        if (rc) return rc;
        if (total_bytes) {
            CU(cudaMemcpyAsync(total_bytes, d_out_off + n, 8, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
        }
        return stream_leave(h, d, st);
    }
    PrepArgs A{d_text, d_text_off, n, op, nullptr, d_out_off, d_out};
    if (n > 0) { LaunchScope ls(h, d, "k_prep_write"); k_prep<true><<<grid, 256, 0, st>>>(A); }
    CU(cudaGetLastError());
    return stream_leave(h, d, st);
}

}  // extern "C"

namespace {

// genztok_bpe_word and, with drop, genztok_bpe_word_dropout after their argument checks.
int bpe_word(genztok_t* h, const uint8_t* word, int64_t word_len, int32_t* piece_cp, int64_t cap, int64_t* n_pieces, const BpeDrop* drop) {
    *n_pieces = 0;
    if (word_len == 0) return GENZTOK_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[0];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = d->stream;
    LaunchScope::cur_stream = st;
    const size_t L = (size_t)word_len;
    CU(d->misc.ensure(L + 64 + (2 * L + 2) * 4));
    uint8_t* dw = d->misc.as<uint8_t>();
    uint32_t* scratch = reinterpret_cast<uint32_t*>(dw + ((L + 63) & ~(size_t)63));
    uint32_t* pieces = scratch + L;
    uint32_t* dn = pieces + L;
    CU(cudaMemcpyAsync(dw, word, L, cudaMemcpyHostToDevice, st));
    if (drop) { LaunchScope ls(h, d, "k_bpe_single_dropout"); k_bpe_single_dropout<<<1, 32, 0, st>>>(d->T, dw, (uint32_t)L, scratch, pieces, dn, *drop); }
    else { LaunchScope ls(h, d, "k_bpe_single"); k_bpe_single<<<1, 32, 0, st>>>(d->T, dw, (uint32_t)L, scratch, pieces, dn); }
    CU(cudaGetLastError());
    uint32_t nn = 0;
    CU(cudaMemcpyAsync(&nn, dn, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *n_pieces = nn;
    if ((int64_t)nn <= cap && piece_cp && nn) {
        CU(cudaMemcpyAsync(piece_cp, pieces, (size_t)nn * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    return GENZTOK_OK;
}

}  // namespace

extern "C" {

// ---- helpers ----------------------------------------------------------------------------------------------
int genztok_bpe_word(genztok_t* h, const uint8_t* word, int64_t word_len, int32_t* piece_cp, int64_t cap, int64_t* n_pieces) {
    if (!h || !n_pieces || word_len < 0) return GENZTOK_E_INVALID;
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    return bpe_word(h, word, word_len, piece_cp, cap, n_pieces, nullptr);
}

// Word 0 of side 0 of a row with key `key` (include/genztok.h): W_0 = mix64(mix64(mix64(seed ^ DROP_K) + key * GOLD) + GOLD).
int genztok_bpe_word_dropout(genztok_t* h, const uint8_t* word, int64_t word_len, double p, uint64_t seed, int64_t key, int32_t* piece_cp, int64_t cap,
                             int64_t* n_pieces) {
    if (!h || !n_pieces || word_len < 0) return GENZTOK_E_INVALID;
    if (!(p >= 0.0 && p <= 1.0)) return fail(h, GENZTOK_E_INVALID, "genztok_bpe_word_dropout: the dropout probability must be in [0, 1] (got %g)", p);
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    const BpeDrop drop{mix64(mix64(mix64(seed ^ DROP_K) + (uint64_t)key * GOLD) + GOLD), (uint64_t)std::floor(p * 4294967296.0)};
    return bpe_word(h, word, word_len, piece_cp, cap, n_pieces, &drop);
}

int genztok_sequence_id(genztok_t* h, const int32_t* ids, int64_t n, int apply_token_type, int8_t* out, int64_t* out_len, int* status) {
    if (!h || n < 0 || !out_len || !status) return GENZTOK_E_INVALID;
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    *out_len = 0; *status = 0;
    if (n == 0) { *status = apply_token_type ? 1 : 0; return GENZTOK_OK; }
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[0];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = d->stream;
    LaunchScope::cur_stream = st;
    CU(d->misc.ensure((size_t)n * 4 + (size_t)n + 64 + 16));
    int32_t* dids = d->misc.as<int32_t>();
    int8_t* dseq = reinterpret_cast<int8_t*>(dids + n);
    int32_t* dlen = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(dids) + (((size_t)n * 5 + 15) & ~(size_t)15));
    uint8_t* dstat = reinterpret_cast<uint8_t*>(dlen + 1);
    CU(cudaMemcpyAsync(dids, ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    PostArgs Q{};
    Q.ids = dids; Q.W = (int32_t)n; Q.n_rows = 1; Q.has_pair = 1; Q.seq = dseq; Q.seq_len = dlen; Q.status = dstat; Q.raw_seq = apply_token_type ? 0 : 1;
    Q.eos_i8 = eos_as_i8(d); Q.pad_i8 = pad_as_i8(d);
    { LaunchScope ls(h, d, "k_post_rows_helper"); k_post_rows<<<1, 32, 0, st>>>(d->T, Q, nullptr); }
    CU(cudaGetLastError());
    int32_t m = 0; uint8_t s8 = 0;
    CU(cudaMemcpyAsync(&m, dlen, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&s8, dstat, 1, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *out_len = m; *status = s8;
    if (out && m > 0) { CU(cudaMemcpyAsync(out, dseq, (size_t)m, cudaMemcpyDeviceToHost, st)); CU(cudaStreamSynchronize(st)); }
    return GENZTOK_OK;
}

int genztok_attention_mask(genztok_t* h, const int32_t* ids, int64_t n, uint8_t* out) {
    if (!h || n < 0) return GENZTOK_E_INVALID;
    if (h->devs.empty()) return fail(h, GENZTOK_E_NODEVICE, "this handle was created without a CUDA device; there is no CPU path");
    if (n == 0) return GENZTOK_OK;
    std::lock_guard<std::mutex> lk(h->mu);
    DeviceCtx* d = h->devs[0];
    CU(cudaSetDevice(d->device));
    cudaStream_t st = d->stream;
    LaunchScope::cur_stream = st;
    CU(d->misc.ensure((size_t)n * 5 + 16));
    int32_t* dids = d->misc.as<int32_t>();
    uint8_t* dm = reinterpret_cast<uint8_t*>(dids + n);
    CU(cudaMemcpyAsync(dids, ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    { LaunchScope ls(h, d, "k_mask_flat"); k_mask_flat<<<(unsigned)std::min<int64_t>((n + 255) / 256, 2048), 256, 0, st>>>(dids, n, d->T.pad, dm); }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, dm, (size_t)n, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return GENZTOK_OK;
}

}  // extern "C"
