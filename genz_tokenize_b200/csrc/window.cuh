// window.cuh -- long documents as overlapping fixed-length windows (HF tokenizers' return_overflowing_tokens with a stride).
//
// The token streams come from the ragged pipeline (k_rows<COUNT> -> k_row_lens -> scan -> k_rows<RAGGED>) run with max_len None
// on each side as single sentences: document d of a stream is [bos] T [eos], untruncated, at off[d].  Then
//   k_window_count   one thread per document: K_d windows from len(A), len(T), max_len W and stride s -> scan -> win_off
//   k_window_rows    one warp per window: the [K, W] planes, row_len / seq_len / row_status and the window -> document map
//   k_post_rows      (row list) pair windows whose content holds a special id: token types from the values (post.cuh)
//
// Window k of a single holds [bos] + T[k(C-s) : k(C-s)+C] + [eos] with C = W - 2.  A pair keeps its first text whole:
// [bos] + A + [eos, eos] + B_k + [eos] with C = W - len(A) - 4; when C - s < 1 the document has one window, its truncated
// pair row.  Every window is then padded to W as tokenize.py:141-182,247-258 pad a row (window 0 is the encode_batch row).
#pragma once
#include "device_common.cuh"
#include "encode.cuh"

namespace gzt {

struct WinArgs {
    const int32_t* ids_a; const int64_t* off_a;   // stream of the text (singles) or of the first text (pairs)
    const int32_t* ids_b; const int64_t* off_b;   // pairs: stream of the second text (NULL for singles)
    int64_t n_docs;
    int32_t W, stride;
    int64_t* count;                               // k_window_count: windows per document
    const int64_t* win_off;                       // [n_docs + 1]
    int64_t n_win;
    int64_t doc_base;                             // added to win_doc (the host form's chunk start)
    int32_t* ids; uint8_t* mask; int8_t* tt; int8_t* seq;   // [n_win, W]; tt / seq may be NULL
    int32_t* row_len; int32_t* seq_len; uint8_t* status;    // [n_win]; seq_len / status may be NULL
    int64_t* win_doc; int32_t* win_start;                   // [n_win]
    uint32_t* fix_list;                           // pair windows for k_post_rows (count at ctr[C_FIX])
    unsigned long long* ctr;                      // the word cache's counters: C_FIX, C_ERR, C_TOKENS
    int8_t eos_i8, pad_i8;
    // offset_mapping (k_window_rows<..., OFFS>): byte (start, end) per token of the streams, aligned with ids_a / ids_b, and the
    // [n_win, W, 2] plane they are cut into
    const int2* offs_a; const int2* offs_b;
    int32_t* offs;
};

// Windows of one document.  L: tokens of the windowed text, LA: tokens of the first text (pairs).
__host__ __device__ __forceinline__ int64_t window_count(int64_t L, int64_t LA, bool pair, int32_t W, int32_t s) {
    const int64_t C = pair ? (int64_t)W - LA - 4 : (int64_t)W - 2;
    if (C - s < 1 || L <= C) return 1;
    return 1 + (L - C + (C - s) - 1) / (C - s);
}

__global__ void __launch_bounds__(256) k_window_count(WinArgs A) {
    const bool pair = A.off_b != nullptr;
    for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d < A.n_docs; d += (int64_t)gridDim.x * blockDim.x) {
        const int64_t LA = A.off_a[d + 1] - A.off_a[d] - 2;
        const int64_t L = pair ? A.off_b[d + 1] - A.off_b[d] - 2 : LA;
        if (LA < 0 || L < 0) atomicAdd(&A.ctr[C_ERR], 1ULL);            // a stream row without its framing
        A.count[d] = window_count(L < 0 ? 0 : L, LA < 0 ? 0 : LA, pair, A.W, A.stride);
    }
}

// One warp per window.  QUAD (W % 4 == 0, planes 16-byte aligned): a lane owns 4 consecutive columns and writes them with one
// 16-byte store of ids and one 4-byte store per byte plane; the pad run needs no loads.  Otherwise a lane owns one column.
// OFFS: the offsets plane too, taken from the streams where the ids are (first text, windowed slice) and (0, 0) elsewhere;
// QUAD writes a lane's 4 columns (32 bytes) with two 16-byte stores.
template <bool QUAD, bool PAIR, bool OFFS = false>
__global__ void __launch_bounds__(256) k_window_rows(DevTables T, WinArgs A) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int32_t W = A.W;
    uint32_t tok_total = 0;
    for (int64_t r = warp; r < A.n_win; r += nwarps) {
        int64_t lo = 0, hi = A.n_docs - 1;                            // the document: last d with win_off[d] <= r
        while (lo < hi) { const int64_t mid = (lo + hi + 1) >> 1; if (A.win_off[mid] <= r) lo = mid; else hi = mid - 1; }
        const int64_t d = lo, k = r - A.win_off[d];
        const int64_t oa = A.off_a[d];
        const int32_t LA = (int32_t)(A.off_a[d + 1] - oa - 2);
        const int64_t ox = PAIR ? A.off_b[d] : oa;
        const int32_t L = PAIR ? (int32_t)(A.off_b[d + 1] - ox - 2) : LA;
        const int32_t C = PAIR ? W - LA - 4 : W - 2;
        const bool whole = PAIR && C - A.stride < 1;                  // one window: the pair row, truncated like encode_batch's
        const int64_t st64 = whole ? 0 : k * (int64_t)(C - A.stride);
        const int32_t st = (int32_t)st64;
        const int32_t len = whole ? L : min(C, L - st);
        if (LA < 0 || L < 0 || k < 0 || k >= window_count(L, LA, PAIR, W, A.stride) || len < 0) {   // win_off does not fit the streams
            if (lane == 0) atomicAdd(&A.ctr[C_ERR], 1ULL);
            continue;
        }
        const int32_t pb = PAIR ? LA + 3 : 1;                         // column of the first windowed token
        const int32_t e = pb + len;                                   // column of the closing </s>
        const int32_t Lf = e + 1;                                     // the window's list before __padding
        const bool trunc = Lf > W;                                    // (whole pair rows only) tokens[:W-1] + [eos]
        const int32_t Lr = trunc ? W : Lf;
        const int32_t* srcA = A.ids_a + oa;                           // srcA[i] = A[i - 1] for columns 1..LA
        const int32_t* srcX = (PAIR ? A.ids_b : A.ids_a) + ox + 1 + st - pb;   // srcX[i] = T[st + i - pb] for columns pb..e-1
        const int2* osrcA = OFFS ? A.offs_a + oa : nullptr;          // the same columns of the offsets streams
        const int2* osrcX = OFFS ? (PAIR ? A.offs_b : A.offs_a) + ox + 1 + st - pb : nullptr;
        auto offset = [&](int32_t i) -> int2 {                       // (0, 0): <s>, </s>, pads, the </s> of a truncated row
            if (i == 0 || (trunc && i == W - 1)) return make_int2(0, 0);
            if (PAIR && i <= LA) return osrcA[i];
            if (PAIR && i < pb) return make_int2(0, 0);
            if (i < e) return osrcX[i];
            return make_int2(0, 0);
        };
        SeqDesc sd;
        if (PAIR) sd = seq_describe(LA, Lf, W);
        bool special = false;
        auto value = [&](int32_t i) -> int32_t {
            if (i == 0) return T.bos;
            if (trunc && i == W - 1) return T.eos;
            if (PAIR && i <= LA) { const int32_t v = srcA[i]; special |= v == T.bos || v == T.eos; return v; }
            if (PAIR && i < pb) return T.eos;
            if (i < e) { const int32_t v = srcX[i]; special |= v == T.bos || v == T.eos; return v; }
            return i == e ? T.eos : T.pad;
        };
        const size_t g0 = (size_t)r * (size_t)W;
        if (QUAD) {
            const uint4 pad4 = make_uint4((uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad);
            for (int32_t i0 = lane * 4; i0 < W; i0 += 128) {
                uint4 v = pad4;
                uint32_t mk = 0;
                if (i0 < Lr) {
                    v = make_uint4((uint32_t)value(i0), (uint32_t)value(i0 + 1), (uint32_t)value(i0 + 2), (uint32_t)value(i0 + 3));
                    mk = (uint32_t)(v.x != (uint32_t)T.pad) | (uint32_t)(v.y != (uint32_t)T.pad) << 8 | (uint32_t)(v.z != (uint32_t)T.pad) << 16 |
                         (uint32_t)(v.w != (uint32_t)T.pad) << 24;
                    tok_total += (uint32_t)__popc(mk);
                }
                st_cs128(A.ids + g0 + i0, v);
                st_cs32(A.mask + g0 + i0, mk);
                if (OFFS) {
                    uint4 o0 = make_uint4(0, 0, 0, 0), o1 = o0;
                    if (i0 < Lr) {
                        const int2 a = offset(i0), b = offset(i0 + 1), c = offset(i0 + 2), d4 = offset(i0 + 3);
                        o0 = make_uint4((uint32_t)a.x, (uint32_t)a.y, (uint32_t)b.x, (uint32_t)b.y);
                        o1 = make_uint4((uint32_t)c.x, (uint32_t)c.y, (uint32_t)d4.x, (uint32_t)d4.y);
                    }
                    st_cs128(A.offs + 2 * (g0 + i0), o0);
                    st_cs128(A.offs + 2 * (g0 + i0) + 4, o1);
                }
                if (PAIR && (A.tt || A.seq)) {
                    uint32_t ttw, sqw;
                    seq_words4(sd, i0, W, A.eos_i8, A.pad_i8, &ttw, &sqw);
                    if (A.tt) st_cs32(A.tt + g0 + i0, ttw);
                    if (A.seq) st_cs32(A.seq + g0 + i0, sqw);
                }
            }
        } else {
            for (int32_t i = lane; i < W; i += 32) {
                const int32_t v = i < Lr ? value(i) : T.pad;
                A.ids[g0 + i] = v;
                A.mask[g0 + i] = (uint8_t)(v != T.pad);
                if (OFFS) reinterpret_cast<int2*>(A.offs)[g0 + i] = i < Lr ? offset(i) : make_int2(0, 0);
                tok_total += (uint32_t)(v != T.pad);
                if (PAIR) {
                    const int32_t sv = i < sd.m ? seq_value(sd, i) : (int32_t)A.pad_i8;
                    if (A.tt) A.tt[g0 + i] = (int8_t)((sd.m == W && i == W - 1) ? (int32_t)A.eos_i8 : sv);
                    if (A.seq) A.seq[g0 + i] = (int8_t)(i < sd.m ? sv : -2);
                }
            }
        }
        special = __any_sync(FULL_MASK, special);
        if (lane == 0) {
            A.row_len[r] = Lr;
            A.win_doc[r] = A.doc_base + d;
            A.win_start[r] = st;
            if (PAIR) {
                if (A.seq_len) A.seq_len[r] = sd.m;
                if (A.status) A.status[r] = (uint8_t)sd.err;
                if (special || !T.specials_distinct) { const unsigned long long j = atomicAdd(&A.ctr[C_FIX], 1ULL); A.fix_list[j] = (uint32_t)r; }
            }
        }
    }
    tok_total = __reduce_add_sync(FULL_MASK, tok_total);
    if (lane == 0 && tok_total) atomicAdd(&A.ctr[C_TOKENS], (unsigned long long)tok_total);
}

}  // namespace gzt
