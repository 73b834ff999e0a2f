// qa.cuh -- extractive question answering over the windows' offset_mapping planes: answer labels from byte (or character) spans,
// and the best answer span per document from a model's start / end logits (HF's postprocess_qa_predictions, top 1, exact).
//
//   k_qa_char_to_byte  a warp per document: character indices of the answer -> byte positions in the document's UTF-8
//   k_qa_labels        a warp per window: (start_positions, end_positions) from the answer's byte span
//   k_qa_spans         a warp per window: the window's best (s, e) and its S[0] + E[0]
//   k_qa_spans_docs    a thread per document: the best window in order, the smallest null score
//
// Context columns come from the offsets alone (window.cuh's layout: every real token spans >= 1 byte, framing and pads are (0, 0)):
// singles, the columns with end > 0; pairs, those after z, the first column >= 1 that is (0, 0).  They form one range [c0, c1)
// whose starts and ends are non-decreasing, so every search below is a search over a monotone predicate.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "device_common.cuh"

namespace gzt {

struct QaArgs {
    const int2* om;                 // [K, W] (start, end)
    int64_t K;
    int32_t W;
    int32_t pair;
    const int64_t* win_off;         // [n + 1]
    int64_t n;
    const int64_t* answers;         // [n][2] byte spans (k_qa_labels)
    int64_t* start; int64_t* end;   // [K] labels
    // k_qa_char_to_byte: character spans in, byte spans out
    const uint8_t* text; const int64_t* text_off; int64_t text_bytes;
    const int64_t* char_answers; int64_t* byte_answers;
    // k_qa_spans
    const float* S; const float* E;  // [K, W]
    int32_t L;                       // max_answer_len
    float* w_score; int32_t* w_s; int32_t* w_e; float* w_null;   // [K] per window (w_s < 0: no candidate)
    float* score; float* null_score; int64_t* window; int32_t* columns; int32_t* span;   // [n], [n], [n], [n][2], [n][2]
    unsigned long long* ctr;         // C_ERR
};

// First c in [lo, hi) with pred(c), or hi; pred false...true on [lo, hi).  32 probes per round: a range of W columns takes
// ceil(log32 W) rounds (two at W <= 1024), each one load per lane.  Warp-uniform arguments.
template <class Pred>
__device__ __forceinline__ int32_t warp_first_true(int32_t lo, int32_t hi, int lane, Pred pred) {
    for (int it = 0; it < 8 && hi - lo > 32; it++) {
        const int32_t step = (hi - lo + 31) / 32;
        const int32_t c = lo + lane * step;
        const unsigned b = __ballot_sync(FULL_MASK, c >= hi || pred(c));
        if (b == 0) { lo += 31 * step + 1; continue; }
        const int k = __ffs(b) - 1;
        if (k == 0) return lo;
        hi = min(hi, lo + k * step);
        lo += (k - 1) * step + 1;
    }
    const int32_t c = lo + lane;
    const unsigned b = __ballot_sync(FULL_MASK, c < hi && pred(c));
    return b ? lo + __ffs(b) - 1 : hi;
}

// The context columns [c0, c1) of one window (c0 == c1: none).  Returns false when the row breaks the layout.
__device__ __forceinline__ bool qa_context(const int2* row, int32_t W, bool pair, int lane, int32_t& c0, int32_t& c1) {
    const int2 f = row[0];
    if (f.x != 0 || f.y != 0) return false;
    if (pair) {
        int32_t z = W;                                               // the </s> after the question: a ballot over 32 columns a round
        for (int32_t b = 1; b < W; b += 32) {
            const int32_t c = b + lane;
            bool zero = false;
            if (c < W) { const int2 o = row[c]; zero = (o.x | o.y) == 0; }
            const unsigned m = __ballot_sync(FULL_MASK, zero);
            if (m) { z = b + __ffs(m) - 1; break; }
        }
        if (z >= W) return false;
        if (z + 1 < W) { const int2 o = row[z + 1]; if ((o.x | o.y) != 0) return false; }   // the second </s>
        c0 = z + 2;
    } else {
        c0 = 1;
    }
    if (c0 >= W || row[c0].y <= 0) { c0 = c1 = min(c0, W); return true; }
    c1 = warp_first_true(c0 + 1, W, lane, [&](int32_t c) { return row[c].y == 0; });
    return true;
}

// Document of window r: the last d with win_off[d] <= r; -1 when win_off does not place r.
__device__ __forceinline__ int64_t qa_doc(const int64_t* win_off, int64_t n, int64_t r) {
    int64_t lo = 0, hi = n - 1;
    while (lo < hi) { const int64_t mid = (lo + hi + 1) >> 1; if (win_off[mid] <= r) lo = mid; else hi = mid - 1; }
    return (n > 0 && win_off[lo] <= r && r < win_off[lo + 1]) ? lo : -1;
}

// Continuation bytes (10xxxxxx) of a 32-bit word, as the top bit of each byte.
__device__ __forceinline__ uint32_t cont_bytes(uint32_t w) { return w & ~(w << 1) & 0x80808080u; }

// Character index -> byte position (the byte of the code point with that index; the character count maps to the byte length,
// larger indices to byte length + the excess, negative ones stay as they are).  A warp per document walks its text 512 bytes a
// round, 16 bytes a lane, counting lead bytes (SWAR + popc), and stops once both indices are placed.
__global__ void __launch_bounds__(256) k_qa_char_to_byte(QaArgs A) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t d = warp; d < A.n; d += nwarps) {
        const int64_t t0 = A.text_off[d], t1 = A.text_off[d + 1];
        const int64_t k[2] = {A.char_answers[2 * d], A.char_answers[2 * d + 1]};
        int64_t out[2] = {k[0] < 0 ? k[0] : -1, k[1] < 0 ? k[1] : -1};
        if (t0 < 0 || t1 < t0 || t1 > A.text_bytes) {
            if (lane == 0) { atomicAdd(&A.ctr[C_ERR], 1ULL); A.byte_answers[2 * d] = 0; A.byte_answers[2 * d + 1] = 0; }
            continue;
        }
        const int64_t kmax = max(k[0], k[1]);
        int64_t cum = 0;                                             // characters before this round
        for (int64_t base = t0 & ~(int64_t)15; base < t1 && cum <= kmax; base += 512) {
            const int64_t p = base + 16 * lane;
            uint32_t lead = 0;                                       // bit j: byte p + j is a lead byte inside [t0, t1)
            if (p < t1 && p + 16 > t0) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(A.text + p));
                const uint32_t w[4] = {v.x, v.y, v.z, v.w};
                for (int q = 0; q < 4; q++) {
                    const uint32_t c = cont_bytes(w[q]);
                    lead |= (uint32_t)((~c >> 7 & 1u) | (~c >> 14 & 2u) | (~c >> 21 & 4u) | (~c >> 28 & 8u)) << (4 * q);
                }
                const int64_t lo = t0 - p, hi = t1 - p;              // keep bytes [lo, hi) of the lane's 16
                if (lo > 0) lead &= ~0u << lo;
                if (hi < 16) lead &= (1u << hi) - 1u;
            }
            const int cnt = __popc(lead);
            int incl = cnt;
            for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += u; }
            const int64_t before = cum + incl - cnt;
            for (int j = 0; j < 2; j++) {
                if (out[j] >= 0 || k[j] < 0) continue;
                if (k[j] >= before && k[j] < before + cnt) {
                    uint32_t m = lead;
                    for (int64_t r = k[j] - before; r > 0; r--) m &= m - 1;
                    out[j] = p - t0 + (__ffs(m) - 1);
                }
            }
            for (int j = 0; j < 2; j++) {                            // broadcast from the lane that placed it
                const unsigned b = __ballot_sync(FULL_MASK, out[j] >= 0 && k[j] >= 0 && k[j] >= before && k[j] < before + cnt);
                if (b) out[j] = __shfl_sync(FULL_MASK, out[j], __ffs(b) - 1);
            }
            cum += __shfl_sync(FULL_MASK, incl, 31);
        }
        for (int j = 0; j < 2; j++)
            if (out[j] < 0 && k[j] >= 0) out[j] = (t1 - t0) + (k[j] - cum);   // at or past the end (all characters counted)
        if (lane == 0) { A.byte_answers[2 * d] = out[0]; A.byte_answers[2 * d + 1] = out[1]; }
    }
}

// Labels: the context columns that overlap [a0, a1) are [s, e] with s the first whose end > a0 and e the last whose start < a1;
// the label is (s, e) when they hold the whole answer, else (0, 0).  A window reads om[0], the question's columns up to z + 1
// (pairs), and ceil(log32 W) rounds of 32 probes for each of c1, s and e.
__global__ void __launch_bounds__(256) k_qa_labels(QaArgs A) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int32_t W = A.W;
    if (blockIdx.x == 0 && threadIdx.x == 0 && (A.n < 0 || A.win_off[0] != 0 || A.win_off[A.n] != A.K)) atomicAdd(&A.ctr[C_ERR], 1ULL);
    for (int64_t r = warp; r < A.K; r += nwarps) {
        const int64_t d = qa_doc(A.win_off, A.n, r);
        int32_t c0 = 0, c1 = 0;
        const int2* row = A.om + (size_t)r * (size_t)W;
        const bool ok = d >= 0 && qa_context(row, W, A.pair != 0, lane, c0, c1);
        int64_t ls = 0, le = 0;
        if (ok && c0 < c1) {
            const int64_t a0 = A.answers[2 * d], a1 = A.answers[2 * d + 1];
            if (a1 > a0) {
                const int32_t s = warp_first_true(c0, c1, lane, [&](int32_t c) { return (int64_t)row[c].y > a0; });
                const int32_t e = warp_first_true(s, c1, lane, [&](int32_t c) { return (int64_t)row[c].x >= a1; }) - 1;
                if (s <= e && (int64_t)row[s].x <= a0 && (int64_t)row[e].y >= a1) { ls = s; le = e; }
            }
        }
        if (lane == 0) {
            if (!ok) atomicAdd(&A.ctr[C_ERR], 1ULL);
            A.start[r] = ls; A.end[r] = le;
        }
    }
}

// Best span of one window.  With the window's rows S, E in shared memory (16-byte loads when W % 4 == 0), the maximum of E over
// [s, s + L - 1] comes from van Herk / Gil-Werman blocks of L columns from c0: P = prefix maxima and Q = suffix maxima inside each
// block (segmented warp scans, 32 columns a round), max E[s..j] = max(Q[s], P[j]).  Float addition is monotone, so
// t(s) = S[s] + max E is the best score with start s; the window's best is the largest t, ties to the smallest s, and its end the
// smallest e in range with S[s] + E[e] == t.  NaN never wins (fmaxf skips it).  O(W + L) per window, any L.
__device__ __forceinline__ void seg_max_scan(float& v, bool head, int lane) {
    bool f = head;
    for (int o = 1; o < 32; o <<= 1) {
        const float vu = __shfl_up_sync(FULL_MASK, v, o);
        const bool fu = __shfl_up_sync(FULL_MASK, (int)f, o) != 0;
        if (lane >= o && !f) { v = fmaxf(v, vu); f = fu; }
    }
}

__global__ void __launch_bounds__(256, 4) k_qa_spans(QaArgs A) {
    extern __shared__ float qa_smem[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int32_t W = A.W, L = A.L;
    float* sS = qa_smem + (size_t)wib * 4 * W;
    float* sE = sS + W;
    float* P = sE + W;
    float* Q = P + W;
    const bool quad = ((W & 3) | ((uintptr_t)A.S & 15) | ((uintptr_t)A.E & 15)) == 0;
    const float NaN = __int_as_float(0x7fc00000);
    for (int64_t r = warp; r < A.K; r += nwarps) {
        const float* gS = A.S + (size_t)r * (size_t)W;
        const float* gE = A.E + (size_t)r * (size_t)W;
        if (quad) {
            for (int32_t c = 4 * lane; c < W; c += 128) {
                *reinterpret_cast<float4*>(sS + c) = __ldcs(reinterpret_cast<const float4*>(gS + c));
                *reinterpret_cast<float4*>(sE + c) = __ldcs(reinterpret_cast<const float4*>(gE + c));
            }
        } else {
            for (int32_t c = lane; c < W; c += 32) { sS[c] = __ldcs(gS + c); sE[c] = __ldcs(gE + c); }
        }
        int32_t c0 = 0, c1 = 0;
        const bool ok = qa_context(A.om + (size_t)r * (size_t)W, W, A.pair != 0, lane, c0, c1);
        __syncwarp();
        // P forward, Q backward, carrying the running maximum from one round of 32 columns to the next
        float carry = NaN;
        for (int32_t b = c0; b < c1; b += 32) {
            const int32_t j = b + lane;
            float v = j < c1 ? sE[j] : NaN;
            const bool head = (j - c0) % L == 0;
            if (lane == 0 && !head) v = fmaxf(v, carry);
            seg_max_scan(v, head || lane == 0, lane);
            if (j < c1) P[j] = v;
            carry = __shfl_sync(FULL_MASK, v, 31);
        }
        carry = NaN;
        for (int32_t b = c1 - 1; b >= c0; b -= 32) {
            const int32_t j = b - lane;
            float v = j >= c0 ? sE[j] : NaN;
            const bool head = j == c1 - 1 || (j - c0) % L == L - 1;
            if (lane == 0 && !head) v = fmaxf(v, carry);
            seg_max_scan(v, head || lane == 0, lane);
            if (j >= c0) Q[j] = v;
            carry = __shfl_sync(FULL_MASK, v, 31);
        }
        __syncwarp();
        bool have = false;
        float bt = 0.f;
        int32_t bs = 0;
        for (int32_t b = c0; b < c1; b += 32) {
            const int32_t s = b + lane;
            if (s >= c1) break;
            const int32_t j = min(s + L - 1, c1 - 1);
            const float mx = (j - c0) / L == (s - c0) / L ? Q[s] : fmaxf(Q[s], P[j]);
            const float ss = sS[s];
            float t = ss + mx;
            if (isnan(t) && ss == -INFINITY && mx == INFINITY) {      // -inf + inf: -inf if some E in range is below +inf
                for (int32_t e = s; e <= j; e++) if (sE[e] < INFINITY) { t = -INFINITY; break; }
            }
            if (!isnan(t) && (!have || t > bt)) { have = true; bt = t; bs = s; }
        }
        for (int o = 16; o > 0; o >>= 1) {
            const bool oh = __shfl_xor_sync(FULL_MASK, (int)have, o) != 0;
            const float ot = __shfl_xor_sync(FULL_MASK, bt, o);
            const int32_t os = __shfl_xor_sync(FULL_MASK, bs, o);
            if (oh && (!have || ot > bt || (ot == bt && os < bs))) { have = true; bt = ot; bs = os; }
        }
        int32_t be = -1;
        if (have) {
            const int32_t j = min(bs + L - 1, c1 - 1);
            const float ss = sS[bs];
            for (int32_t b = bs; b <= j; b += 32) {
                const int32_t e = b + lane;
                const unsigned m = __ballot_sync(FULL_MASK, e <= j && ss + sE[e] == bt);
                if (m) { be = b + __ffs(m) - 1; break; }
            }
        }
        if (lane == 0) {
            if (!ok) atomicAdd(&A.ctr[C_ERR], 1ULL);
            const bool found = ok && have && be >= 0;
            A.w_score[r] = found ? bt : -INFINITY;
            A.w_s[r] = found ? bs : -1;
            A.w_e[r] = found ? be : -1;
            A.w_null[r] = sS[0] + sE[0];
        }
        __syncwarp();
    }
}

// A thread per document: its windows in order (ties keep the earlier window), the null score as the fminf over them.
__global__ void __launch_bounds__(256) k_qa_spans_docs(QaArgs A) {
    for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; d < A.n; d += (int64_t)gridDim.x * blockDim.x) {
        int64_t w0 = A.win_off[d], w1 = A.win_off[d + 1];
        if (w0 < 0 || w1 < w0 || w1 > A.K) { atomicAdd(&A.ctr[C_ERR], 1ULL); w1 = w0 = 0; }
        float best = -INFINITY, nul = __int_as_float(0x7fc00000);
        int64_t bw = -1;
        for (int64_t i = w0; i < w1; i++) {
            nul = fminf(nul, A.w_null[i]);
            if (A.w_s[i] >= 0 && (bw < 0 || A.w_score[i] > best)) { best = A.w_score[i]; bw = i; }
        }
        int2 cols = make_int2(0, 0), sp = make_int2(0, 0);
        if (bw >= 0) {
            cols = make_int2(A.w_s[bw], A.w_e[bw]);
            const int2* row = A.om + (size_t)bw * (size_t)A.W;
            sp = make_int2(row[cols.x].x, row[cols.y].y);
        }
        A.score[d] = best;
        A.null_score[d] = nul;
        A.window[d] = bw;
        reinterpret_cast<int2*>(A.columns)[d] = cols;
        reinterpret_cast<int2*>(A.span)[d] = sp;
    }
}

}  // namespace gzt
