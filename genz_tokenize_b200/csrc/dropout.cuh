// dropout.cuh -- BPE-dropout (Provilkov et al., 2020) for fixed-layout encodes: the ids of every text with each merge skipped at
// random, per occurrence of a word.  include/genztok.h states the rule and the hash.
//
// A word's segmentation changes from one occurrence to the next, so the word cache cannot serve it: every word runs its own merge
// loop, straight from the text.  Per chunk the device runs
//   k_dropout_stream   one warp per (document, side): the \S+\n? words of the text (encode.cuh's classifiers), and per word
//                      bpe_symbols + the dropout rounds of bpe.cuh, one word after another; the first `cap` (= max_len) ids of
//                      the text go to slot d of the side's stream, its length to len[d].  The walk stops once the text has cap
//                      ids: the reference cut never shows more of a text.
//   k_dropout_rows     (window.cuh) one warp per row: the reference's row, cut and padded, from the two capped streams
//   k_post_rows        (row list) pair rows whose content holds a special id
// Stream sizes are known before the launch (n * (cap + 2) per side), so nothing is read back.
#pragma once
#include "bpe.cuh"
#include "device_common.cuh"
#include "encode.cuh"

namespace gzt {

static const uint64_t DROP_K = 0x6270655F64726F70ULL;   // "bpe_drop"
static const int DROP_WIN = 512;                         // bytes a warp classifies per step: 16 per lane
static const int DROP_WORDS = DROP_WIN / 2;              // word starts (and ends) one step can hold

struct DropArgs {
    Side a, b;                          // b.off == NULL: single sentences
    int64_t n;
    int32_t cap;                        // ids kept per text; slot d of a stream is [d * (cap + 2), (d + 1) * (cap + 2)), ids from entry 1
    uint64_t s0, thr;                   // mix64(seed ^ DROP_K), floor(p * 2^32)
    const int64_t* row_keys;            // [n]; NULL: key_base + d
    int64_t key_base;
    int32_t* ids_a; int32_t* ids_b;     // the streams
    int32_t* len_a; int32_t* len_b;     // [n] ids in each slot (<= cap)
    // words longer than BPE_SMEM_SYMS: symbols at scratch[q], ranks at scratch[nbytes + q], q = the word's byte position in the
    // chunk (side a's b_base bytes first, then side b's: nbytes in all)
    uint32_t* scratch;
    int64_t b_base, nbytes;
    unsigned long long* ctr;            // the word cache's counters: C_ERR counts documents whose offsets do not fit the side's bytes
};

__global__ void __launch_bounds__(256) k_dropout_stream(DevTables T, DropArgs A) {
    __shared__ uint32_t sm_sym[8][BPE_SMEM_SYMS];
    __shared__ uint32_t sm_rank[8][BPE_SMEM_SYMS];
    __shared__ uint32_t sm_dirty[8][64];
    __shared__ uint16_t sm_st[8][DROP_WORDS], sm_en[8][DROP_WORDS];   // word starts / ends of the current step, in byte order
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t nwork = A.b.off ? 2 * A.n : A.n;
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < nwork; w += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int side = w >= A.n ? 1 : 0;
        const int64_t d = w - side * A.n;
        const int64_t* off = side ? A.b.off : A.a.off;
        const int64_t f0 = off[0];
        int64_t o0 = off[d] - f0, o1 = off[d + 1] - f0;               // from the side's first byte
        // a document must lie inside its side's bytes (the text and the long-word scratch are addressed from there); one that does
        // not is counted (genztok_check_errors) and walked as an empty text: it gets no ids
        if (o0 < 0 || o1 < o0 || o1 > (side ? A.nbytes - A.b_base : A.b_base) || o1 - o0 > (int64_t)INT32_MAX - 64) {
            if (lane == 0) atomicAdd(&A.ctr[C_ERR], 1ULL);
            o0 = o1 = 0;
        }
        const uint8_t* tb = (side ? A.b.bytes : A.a.bytes) + ((o0 + f0) & ~(int64_t)15);   // 16-byte aligned; the text is [S0, E) from here
        const int32_t S0 = (int32_t)((o0 + f0) & 15), E = S0 + (int32_t)(o1 - o0);
        const int32_t doff[2] = {S0, E};
        uint32_t* scr = A.scratch + (side ? A.b_base : 0) + o0 - S0;   // scr + p: the word at p
        int32_t* out = (side ? A.ids_b : A.ids_a) + d * (int64_t)(A.cap + 2) + 1;
        const uint64_t R = mix64(A.s0 + (uint64_t)(A.row_keys ? A.row_keys[d] : A.key_base + d) * GOLD);
        uint32_t j = 0;                                               // words met so far
        int32_t pos = 0;                                              // ids written so far
        auto word = [&](int32_t st, int32_t en) {                     // [st, en): \S+ ; the \n? is added here (tokenize.py:106)
            if (en < E && tb[en] == 0x0A) en++;
            const uint32_t len = (uint32_t)(en - st);
            const BpeDrop D{mix64(R + (2ull * j + (uint64_t)side + 1ull) * GOLD), A.thr};
            j++;
            const bool big = len > (uint32_t)BPE_SMEM_SYMS;
            uint32_t* S = big ? scr + st : sm_sym[wib];
            uint32_t n = bpe_symbols(T, tb + st, len, S, lane);
            if (n <= 32) n = bpe_rounds(T, S, n, lane, D);
            else n = bpe_rounds_cached(T, S, big ? scr + A.nbytes + st : sm_rank[wib], n, lane, sm_dirty[wib], D);
            const uint32_t keep = min(n, (uint32_t)(A.cap - pos));
            for (uint32_t i = lane; i < keep; i += 32) out[pos + (int32_t)i] = sym_to_id(T, S[i], i == n - 1);
            pos += (int32_t)keep;
            __syncwarp();                                             // S is read above before the next word writes it
        };
        int32_t open = -1;                                            // a word whose end is in a later step
        uint32_t prev_ws = 1, spill = 0;                              // the byte before this step is whitespace; multi-byte spill
        for (int32_t base = 0; base < E && pos < A.cap; base += DROP_WIN) {
            const int32_t a = base + 16 * lane;
            const uint32_t ws = a < E ? classify16(ldg128(tb + a), tb, a, S0, E, doff, 1) : 0xFFFFu;   // outside the text: whitespace
            const uint32_t up = __shfl_up_sync(FULL_MASK, ws, 1);
            const uint32_t wsm = (ws | (lane ? (up >> 16) & 3u : spill)) & 0xFFFFu;
            const uint32_t upm = __shfl_up_sync(FULL_MASK, wsm, 1);
            const uint32_t wsb = ((wsm << 1) | (lane ? (upm >> 15) & 1u : prev_ws)) & 0xFFFFu;   // bit k: byte k - 1 is whitespace
            const uint32_t starts = ~wsm & wsb & 0xFFFFu, ends = wsm & ~wsb & 0xFFFFu;
            spill = __shfl_sync(FULL_MASK, (ws >> 16) & 3u, 31);
            prev_ws = __shfl_sync(FULL_MASK, (wsm >> 15) & 1u, 31);
            uint32_t xs = __popc(starts), xe = __popc(ends);
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t ts = __shfl_up_sync(FULL_MASK, xs, o), te = __shfl_up_sync(FULL_MASK, xe, o);
                if (lane >= o) { xs += ts; xe += te; }
            }
            const uint32_t ns = __shfl_sync(FULL_MASK, xs, 31), ne = __shfl_sync(FULL_MASK, xe, 31);
            xs -= __popc(starts); xe -= __popc(ends);
            for (uint32_t m = starts; m; m &= m - 1) sm_st[wib][xs++] = (uint16_t)(16 * lane + __ffs(m) - 1);
            for (uint32_t m = ends; m; m &= m - 1) sm_en[wib][xe++] = (uint16_t)(16 * lane + __ffs(m) - 1);
            __syncwarp();
            // starts and ends alternate in byte order: the k-th end of the step closes the open word, then the starts in turn
            for (uint32_t ks = 0, ke = 0; pos < A.cap;) {
                int32_t st = open;
                if (st < 0) { if (ks >= ns) break; st = base + sm_st[wib][ks++]; }
                if (ke >= ne) { open = st; break; }
                open = -1;
                word(st, base + sm_en[wib][ke++]);
            }
            __syncwarp();                                             // the lists are read before the next step writes them
        }
        if (open >= 0 && pos < A.cap) word(open, E);
        if (lane == 0) (side ? A.len_b : A.len_a)[d] = pos;
    }
}

}  // namespace gzt
