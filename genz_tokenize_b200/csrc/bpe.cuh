// bpe.cuh -- the BPE merge loop, one warp per distinct word (north_star step 3).
//
// Replaces tokenize.py:62-101 (bpe) and :270-278 (get_pairs) for words that the device word cache
// has not seen yet, and :99-100,:120-121 (piece -> id).  The reference's round structure is kept
// exactly: in every round take the lowest-rank pair among the CURRENT adjacent pairs, merge all of
// its non-overlapping occurrences left to right, stop when no pair has a rank or one symbol is left.
// Symbols are integer ids of the strings the reference would hold (host_tables.hpp).
#pragma once
#include "device_common.cuh"

namespace gzt {

static const int BPE_SMEM_SYMS = 128;        // words up to 128 bytes are merged in shared memory
static const uint32_t CP_INVALID = 0xFFFFFFFEu;

// UTF-8 bytes -> initial symbols (tokenize.py:63-64).  S needs room for `len` entries. Returns #symbols.
__device__ __forceinline__ uint32_t bpe_symbols(const DevTables& T, const uint8_t* key, uint32_t len, uint32_t* S, int lane) {
    uint32_t n = 0, last_fin = SYM_NONE;
    for (uint32_t base = 0; base < len; base += 32) {
        uint32_t j = base + lane;
        uint32_t b = j < len ? key[j] : 0;
        bool lead = j < len && (((b & 0xC0) != 0x80) || j == 0);
        uint32_t m = __ballot_sync(FULL_MASK, lead);
        uint32_t mid = SYM_NONE, fin = SYM_NONE;
        if (lead) {
            int expect = b < 0x80 ? 1 : (b & 0xE0) == 0xC0 ? 2 : (b & 0xF0) == 0xE0 ? 3 : (b & 0xF8) == 0xF0 ? 4 : 0;
            uint32_t cp = expect == 1 ? b : expect == 2 ? (b & 0x1F) : expect == 3 ? (b & 0x0F) : (b & 0x07);
            int got = 1;
            for (uint32_t k = j + 1; k < len && got < 5; k++) {
                uint32_t c = key[k];
                if ((c & 0xC0) != 0x80) break;
                cp = (cp << 6) | (c & 0x3F);
                got++;
            }
            if (expect == 0 || got != expect) cp = CP_INVALID;
            if (cp != CP_INVALID) cp_symbols(T, cp, &mid, &fin);
            S[n + __popc(m & ((1u << lane) - 1))] = mid;
        }
        if (m) last_fin = __shfl_sync(FULL_MASK, fin, 31 - __clz(m));
        n += __popc(m);
    }
    __syncwarp();
    if (lane == 0 && n > 0) S[n - 1] = last_fin;   // the last code point carries "</w>"
    __syncwarp();
    return n;
}

// The merge rounds (tokenize.py:69-98) on S[0..n). Returns the new length.
__device__ __forceinline__ uint32_t bpe_rounds(const DevTables& T, uint32_t* S, uint32_t n, int lane) {
    for (uint32_t round = 0, n0 = n; n > 1 && round <= n0; round++) {   // every round removes >= 1 symbol
        // ---- bigram = min(pairs, key=rank)  (:70-71)
        uint32_t best = 0xFFFFFFFFu, ba = 0, bb = 0, bm = 0;
        for (uint32_t base = 0; base + 1 < n; base += 32) {
            uint32_t i = base + lane;
            if (i + 1 < n) {
                uint32_t a = S[i], b = S[i + 1], mg;
                uint32_t r = pair_rank(T, a, b, &mg);
                if (r < best) { best = r; ba = a; bb = b; bm = mg; }
            }
        }
        uint32_t gbest = __reduce_min_sync(FULL_MASK, best);
        if (gbest == 0xFFFFFFFFu) break;                       // `if bigram not in self.bpe_ranks: break` (:72-73)
        int src = __ffs(__ballot_sync(FULL_MASK, best == gbest)) - 1;   // ranks are unique per pair
        ba = __shfl_sync(FULL_MASK, ba, src);
        bb = __shfl_sync(FULL_MASK, bb, src);
        bm = __shfl_sync(FULL_MASK, bm, src);
        // ---- merge every non-overlapping (first, second) scanning left to right (:75-92)
        uint32_t out = 0, carry = 0;   // carry: element `base` was consumed by a merge selected at base-1
        for (uint32_t base = 0; base < n; base += 32) {
            uint32_t i = base + lane;
            uint32_t a = i < n ? S[i] : SYM_NONE;
            uint32_t b = i + 1 < n ? S[i + 1] : SYM_NONE;
            bool match = (i + 1 < n) && a == ba && b == bb;
            uint32_t m = __ballot_sync(FULL_MASK, match);
            uint32_t sel;
            if (ba == bb) {
                // runs of equal symbols: greedy picks every second match from the run start (a a a -> aa a)
                uint32_t below = ~m & ((1u << lane) - 1);
                int start = below ? 32 - __clz(below) : 0;           // first index of the run of matches ending at me
                bool odd = ((lane - start) & 1) != 0;
                bool pick = match && ((start == 0 && carry) ? odd : !odd);
                sel = __ballot_sync(FULL_MASK, pick);
            } else {
                sel = m;
            }
            uint32_t consumed = (sel << 1) | carry;
            carry = sel >> 31;
            uint32_t valid = (n - base >= 32) ? FULL_MASK : ((1u << (n - base)) - 1);
            uint32_t keep = valid & ~consumed;
            uint32_t v = ((sel >> lane) & 1) ? bm : a;
            __syncwarp();                                            // all loads of this window done before stores
            if ((keep >> lane) & 1) S[out + __popc(keep & ((1u << lane) - 1))] = v;
            out += __popc(keep);
        }
        __syncwarp();
        n = out;                                                     // `if len(word) == 1: break` (:95-96) via loop condition
    }
    return n;
}

// The same rounds for words of more than 32 symbols, with the rank of every adjacent pair kept in R between rounds: a round
// reads the ranks (no table look-ups), merges, and then looks up only the pairs next to the symbols it has just made -- two per
// merge site instead of one per symbol.  A 1,200-byte token costs ~40 look-up round trips per round the plain loop above; here ~2.
// R needs n entries; dlist is a 64-entry scratch list in shared memory.  (tokenize.py:69-98: the same rounds, the same result.)
static const uint32_t RANK_NONE = 0xFFFFFFFFu, RANK_DIRTY = 0xFFFFFFFEu;
__device__ __forceinline__ uint32_t bpe_rounds_cached(const DevTables& T, uint32_t* S, uint32_t* R, uint32_t n, int lane, uint32_t* dlist) {
    for (uint32_t i = lane; i < n; i += 32) { uint32_t mg; R[i] = i + 1 < n ? pair_rank(T, S[i], S[i + 1], &mg) : RANK_NONE; }
    __syncwarp();
    for (uint32_t round = 0, n0 = n; n > 1 && round <= n0; round++) {
        // ---- bigram = min(pairs, key=rank)  (:70-71)
        uint32_t best = RANK_NONE, bi = 0;
        for (uint32_t i = lane; i + 1 < n; i += 32) { const uint32_t r = R[i]; if (r < best) { best = r; bi = i; } }
        const uint32_t gbest = __reduce_min_sync(FULL_MASK, best);
        if (gbest >= RANK_DIRTY) break;                          // `if bigram not in self.bpe_ranks: break` (:72-73)
        const int src = __ffs(__ballot_sync(FULL_MASK, best == gbest)) - 1;
        bi = __shfl_sync(FULL_MASK, bi, src);
        const uint32_t ba = S[bi], bb = S[bi + 1];
        uint32_t bm = 0;
        pair_rank(T, ba, bb, &bm);
        // ---- merge every non-overlapping (first, second) scanning left to right (:75-92); S and R are compacted together
        uint32_t out = 0, carry = 0, nd = 0;
        bool overflow = false;
        uint32_t prev_idx = 0; bool prev_plain = false;          // the last kept element of the window before: its new index, and "not itself merged"
        for (uint32_t base = 0; base < n; base += 32) {
            const uint32_t i = base + lane;
            const uint32_t a = i < n ? S[i] : SYM_NONE;
            const uint32_t r = i < n ? R[i] : RANK_NONE;
            const bool match = (i + 1 < n) && r == gbest;
            const uint32_t m = __ballot_sync(FULL_MASK, match);
            uint32_t sel;
            if (ba == bb) {                                      // runs of equal symbols: every second match from the run start (a a a -> aa a)
                const uint32_t below = ~m & ((1u << lane) - 1);
                const int start = below ? 32 - __clz(below) : 0;
                const bool odd = ((lane - start) & 1) != 0;
                const bool pick = match && ((start == 0 && carry) ? odd : !odd);
                sel = __ballot_sync(FULL_MASK, pick);
            } else sel = m;
            const uint32_t consumed = (sel << 1) | carry;
            const uint32_t valid = (n - base >= 32) ? FULL_MASK : ((1u << (n - base)) - 1);
            const uint32_t keep = valid & ~consumed;
            // a kept element's pair changes when it is a merged symbol or the element behind it is: sel(i) | sel(i + 1); the
            // bit for lane 31 comes with the next window (below)
            const uint32_t dirty = keep & (sel | (sel >> 1));
            const uint32_t k = out + __popc(keep & ((1u << lane) - 1));
            const uint32_t v = ((sel >> lane) & 1) ? bm : a;
            __syncwarp();                                        // all loads of this window done before the stores
            if ((keep >> lane) & 1) { S[k] = v; R[k] = ((dirty >> lane) & 1) ? RANK_DIRTY : r; }
            uint32_t dm = dirty;
            if ((sel & 1u) && prev_plain) {                      // the element before this window's first merge: dirty after all
                if (lane == 0) R[prev_idx] = RANK_DIRTY;
                if (nd < 64) { if (lane == 0) dlist[nd] = prev_idx; nd++; } else overflow = true;
            }
            const uint32_t cnt = __popc(dm);
            if (nd + cnt <= 64) { if ((dm >> lane) & 1) dlist[nd + __popc(dm & ((1u << lane) - 1))] = k; nd += cnt; }
            else overflow = true;
            const uint32_t nk = __popc(keep);
            if (keep) { const int hi_lane = 31 - __clz(keep); prev_idx = out + nk - 1; prev_plain = !((sel >> hi_lane) & 1); }
            out += nk;
            carry = sel >> 31;
        }
        __syncwarp();
        n = out;                                                 // `if len(word) == 1: break` (:95-96) via the loop condition
        // ---- the ranks of the pairs that changed
        if (!overflow) {
            for (uint32_t j = lane; j < nd; j += 32) { const uint32_t k = dlist[j]; uint32_t mg; R[k] = k + 1 < n ? pair_rank(T, S[k], S[k + 1], &mg) : RANK_NONE; }
        } else {
            for (uint32_t i = lane; i < n; i += 32) if (R[i] == RANK_DIRTY) { uint32_t mg; R[i] = i + 1 < n ? pair_rank(T, S[i], S[i + 1], &mg) : RANK_NONE; }
        }
        if (lane == 0 && n > 0) R[n - 1] = RANK_NONE;
        __syncwarp();
    }
    return n;
}

// symbol -> vocab id: non-final symbols are looked up as S+"@@", the final one as S[:-4] (:99-100,:120-121)
__device__ __forceinline__ int32_t sym_to_id(const DevTables& T, uint32_t s, bool final_sym) {
    if (s == SYM_NONE) return T.unk;
    return final_sym ? T.id_fin[s] : T.id_cont[s];
}

// Position of the k-th (0-based) set bit of m; m has more than k set bits.
__device__ __forceinline__ uint32_t nth_set_bit(uint32_t m, uint32_t k) {
    for (uint32_t t = 0; t < k; t++) m &= m - 1;
    return (uint32_t)__ffs(m) - 1u;
}

// offset_mapping: byte length of each of the n final pieces S[0..n) of the word key[0..len), into out[0..n).  Piece i holds the
// code points k_bpe_single reports for it (sym_ncp, less the 4 of "</w>" on the last piece; an unknown code point is one), cut
// where bpe_symbols cuts them (at every byte that is not a continuation byte, and at byte 0).  Lane i of each group of 32
// pieces finds the byte of its past-the-end code point by counting lead bytes from the group's first byte.  All 32 lanes
// call this; lane i reads only S[i + 32k] (S may alias the arena entry that k_bpe_pending then converts in place).
__device__ __noinline__ void bpe_piece_lens(const uint32_t* sym_ncp, const uint8_t* key, uint32_t len, const uint32_t* S, uint32_t n, uint16_t* out) {
    const int lane = threadIdx.x & 31;
    uint32_t p = 0;                                              // byte of the group's first code point
    for (uint32_t base = 0; base < n; base += 32) {
        const uint32_t i = base + lane;
        uint32_t e = i < n ? (S[i] == SYM_NONE ? 1u : sym_ncp[S[i]] - (i == n - 1 ? 4u : 0u)) : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(FULL_MASK, e, o); if (lane >= o) e += t; }
        // e: code points of the group up to my piece's end; the byte where that code point starts ends my piece
        const uint32_t G = __shfl_sync(FULL_MASK, e, 31);
        uint32_t be = len;                                       // (a code point past the word's last one starts at len)
        for (uint32_t q = p, seen = 0; q < len && seen <= G; q += 32) {
            const uint32_t j = q + lane;
            const uint32_t m = __ballot_sync(FULL_MASK, j < len && (((key[j] & 0xC0) != 0x80) || j == 0));
            const uint32_t c = __popc(m);
            if (e >= seen && e < seen + c) be = q + nth_set_bit(m, e - seen);
            seen += c;
        }
        uint32_t bs = __shfl_up_sync(FULL_MASK, be, 1);          // my piece starts where the one before ends
        if (lane == 0) bs = p;
        if (i < n) out[i] = (uint16_t)(be - bs);
        p = __shfl_sync(FULL_MASK, be, 31);
    }
    __syncwarp();
}

// One warp per pending cache slot.  plen (offset_mapping; NULL when no call on this device has asked for offsets): the byte
// length of every piece of a VAL_MULTI entry, at the index of its id in tok_arena.
__global__ void __launch_bounds__(256) k_bpe_pending(DevTables T, WordCache C, uint16_t* plen) {
    pdl_wait(); pdl_trigger();
    __shared__ uint32_t sm_sym[8][BPE_SMEM_SYMS];
    __shared__ uint32_t sm_rank[8][BPE_SMEM_SYMS];
    __shared__ uint32_t sm_dirty[8][64];
    __shared__ __align__(16) uint8_t sm_key[8][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint64_t npend = C.ctr[C_PENDING];
    if (npend > C.pending_cap) npend = C.pending_cap;
    // no more warps than words draw tickets (in steady state nothing is pending: thousands of warps would queue up on one atomic)
    if ((((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) >= npend) return;
    // words are handed out by a ticket: a 1,200-byte token costs a thousand times a syllable, a fixed assignment of words to
    // warps would leave the kernel waiting for the warp that drew several of them
    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(&C.ctr[C_TICKET], 1ULL);
        w = __shfl_sync(FULL_MASK, w, 0);
        if (w >= npend) break;
        Slot* s = &C.slots[C.pending[w]];
        const uint32_t len = s->len;
        const uint8_t* key;
        if (len <= KEY_INLINE) {
            if (lane < 3) reinterpret_cast<uint64_t*>(sm_key[wib])[lane] = lane == 0 ? s->k0 : lane == 1 ? s->k1 : s->k2;
            __syncwarp();
            key = sm_key[wib];
        } else {
            key = C.key_arena + s->k0;
        }
        uint32_t* S;
        uint32_t scratch_off = 0;
        const bool big = len > (uint32_t)BPE_SMEM_SYMS;
        if (big) {   // long word: work in place in the token arena (capacity reserved by the chunk guard); entry 0 = count
            if (lane == 0) scratch_off = (uint32_t)atomicAdd(&C.ctr[C_TOKS], (unsigned long long)len + 1);
            scratch_off = __shfl_sync(FULL_MASK, scratch_off, 0);
            S = C.tok_arena + scratch_off + 1;
        } else {
            S = sm_sym[wib];
        }
        uint32_t n = bpe_symbols(T, key, len, S, lane);
        if (n <= 32) n = bpe_rounds(T, S, n, lane);
        else {
            uint32_t* R = sm_rank[wib];
            if (big) {   // its ranks live in the per-call scratch (as many entries as the word has bytes: the guard reserved the chunk's size)
                uint32_t ro = 0;
                if (lane == 0) ro = (uint32_t)atomicAdd(&C.ctr[C_SCRATCH], (unsigned long long)len);
                ro = __shfl_sync(FULL_MASK, ro, 0);
                R = C.rank_scratch + ro;
                if ((uint64_t)ro + len > C.rank_cap) { if (lane == 0) atomicAdd(&C.ctr[C_ERR], 1ULL); R = nullptr; }
            }
            n = R ? bpe_rounds_cached(T, S, R, n, lane, sm_dirty[wib]) : bpe_rounds(T, S, n, lane);
        }
        uint32_t val;
        // VAL_SINGLE promises "one token that is none of <s>, </s>, <pad>": a word that IS one of those ids (the text "</s>")
        // is stored as a list of one, so that the row kernels meet it on their general path and never test ids in the common one
        const int32_t id1 = n == 1 ? sym_to_id(T, S[0], true) : -1;
        if (n == 1 && id1 != T.bos && id1 != T.eos && id1 != T.pad) {
            val = VAL_SINGLE | ((uint32_t)id1 & VAL_PAYLOAD);
        } else {
            uint32_t off = scratch_off;
            if (!big) {
                if (lane == 0) off = (uint32_t)atomicAdd(&C.ctr[C_TOKS], (unsigned long long)n + 1);
                off = __shfl_sync(FULL_MASK, off, 0);
            }
            // piece lengths first: for a long word S is the arena entry the loop below converts in place
            if (plen) bpe_piece_lens(T.sym_ncp, key, len, S, n, plen + off + 1);
            // (for a long word S aliases tok_arena + off + 1: each lane converts its own entries in place;
            //  no warp-level sync may sit inside this loop, its trip count differs per lane)
            for (uint32_t i = lane; i < n; i += 32) C.tok_arena[off + 1 + i] = (uint32_t)sym_to_id(T, S[i], i == n - 1);
            if (lane == 0) C.tok_arena[off] = n;
            val = VAL_MULTI | off;
        }
        __syncwarp();
        if (lane == 0) s->val = val;
        __syncwarp();
    }
}

// Tokenize.bpe(token) helper (tokenize.py:62-101): one word in `word`, result = code points per piece.
__global__ void k_bpe_single(DevTables T, const uint8_t* word, uint32_t len, uint32_t* scratch, uint32_t* piece_ncp, uint32_t* n_out) {
    const int lane = threadIdx.x & 31;
    uint32_t n = bpe_symbols(T, word, len, scratch, lane);
    n = bpe_rounds(T, scratch, n, lane);
    for (uint32_t i = lane; i < n; i += 32) piece_ncp[i] = scratch[i] == SYM_NONE ? 1u : T.sym_ncp[scratch[i]] - ((i == n - 1) ? 4u : 0u);
    if (lane == 0) *n_out = n;
}

}  // namespace gzt
