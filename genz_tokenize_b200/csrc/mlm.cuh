// mlm.cuh -- masked-language-model inputs and labels from a fixed-layout id plane (HF's DataCollatorForLanguageModeling recipe,
// token or whole-word selection), one pass over the plane.  The semantics are stated in include/genztok.h.
//
//   k_mlm_mask<WHOLE_WORD>  a warp per row, 128 columns a step, 4 consecutive columns a lane (one 16-byte load of ids, 16 + 32
//                           bytes of stores when the row and the pointers allow it, else 4 scalar accesses).  Whole words: a
//                           column starts a group unless the column before it holds a continuation id (a vocab string ending in
//                           "@@"); the lane's previous column comes from a ballot of the lanes' last columns and, for lane 0,
//                           a carry from the step before.  The selection hash runs once per group, at its start; the decision
//                           reaches the group's other columns through a ballot of "the lane has a start" and of the decision
//                           of its last start, plus the same kind of carry.  The action hash runs only at selected columns.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "device_common.cuh"

namespace gzt {

static const uint64_t MLM_K = 0x6D6C6D5F6D61736BULL;   // "mlm_mask"

struct MlmArgs {
    const int32_t* ids;               // [n, W]
    int64_t n;
    int32_t W;
    const int64_t* row_keys;          // [n] or NULL: row r has key r
    uint64_t s0;                      // mix64(seed ^ MLM_K)
    uint64_t t_sel, t_mask, t_mask_rand;   // thresholds on the top 32 bits of a hash (up to 2^32)
    const uint32_t* cont;             // bitset over [0, n_ids): the id continues into the next piece
    const int32_t* repl;              // [m] the ids random replacement draws from
    uint32_t m;
    int32_t n_ids;
    int32_t pad, bos, eos, msk, unk;
    int32_t* out;                     // [n, W] masked ids
    int64_t* labels;                  // [n, W]
};

template <bool WHOLE_WORD>
__global__ void __launch_bounds__(256) k_mlm_mask(MlmArgs A) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int32_t W = A.W;
    const bool quad = ((W & 3) | ((uintptr_t)A.ids & 15) | ((uintptr_t)A.out & 15) | ((uintptr_t)A.labels & 15)) == 0;
    const unsigned below = (1u << lane) - 1u;
    for (int64_t r = warp; r < A.n; r += nwarps) {
        const uint64_t key = A.row_keys ? (uint64_t)__ldg(&A.row_keys[r]) : (uint64_t)r;
        const uint64_t R = mix64(A.s0 + key * GOLD);
        const int32_t* src = A.ids + (size_t)r * (size_t)W;
        int32_t* dst = A.out + (size_t)r * (size_t)W;
        int64_t* lab = A.labels + (size_t)r * (size_t)W;
        uint32_t carry_cont = 0, carry_dec = 0;                 // the step before: its last column continues / its last group's decision
        for (int32_t b = 0; b < W; b += 128) {
            const int32_t c0 = b + 4 * lane;
            int32_t x[4];
            if (quad) {
                if (c0 < W) { const int4 v = __ldcs(reinterpret_cast<const int4*>(src + c0)); x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; }
                else x[0] = x[1] = x[2] = x[3] = -1;
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++) x[k] = c0 + k < W ? __ldcs(src + c0 + k) : -1;
            }
            uint32_t elig = 0, cont = 0;                         // bit k: column c0 + k
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int32_t v = x[k];
                const bool in = v >= 0 && v < A.n_ids;
                if (in && v != A.pad && v != A.bos && v != A.eos && v != A.msk && v != A.unk) elig |= 1u << k;
                if (WHOLE_WORD && in && ((__ldg(&A.cont[v >> 5]) >> (v & 31)) & 1u)) cont |= 1u << k;
            }
            uint32_t sel = 0;                                    // bit k: column c0 + k is selected
            if (WHOLE_WORD) {
                const unsigned last_cont = __ballot_sync(FULL_MASK, (cont >> 3) & 1u);
                const uint32_t prev = lane ? (last_cont >> (lane - 1)) & 1u : carry_cont;
                const uint32_t start = ~((cont << 1) | prev) & 0xFu;   // bit k: column c0 + k starts a group
                uint32_t dec = 0;                                // decisions at the starts
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (((start >> k) & 1u) && (((elig | cont) >> k) & 1u) &&   // a group of one ineligible column needs no decision
                        (mix64(R + (2ull * (uint64_t)(c0 + k) + 1ull) * GOLD) >> 32) < A.t_sel)
                        dec |= 1u << k;
                const uint32_t last_start = start ? 31u - __clz(start) : 0u;
                const unsigned has = __ballot_sync(FULL_MASK, start != 0);
                const unsigned ldec = __ballot_sync(FULL_MASK, (dec >> last_start) & 1u);
                const unsigned before = has & below;
                uint32_t cur = before ? (ldec >> (31 - __clz(before))) & 1u : carry_dec;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    if ((start >> k) & 1u) cur = (dec >> k) & 1u;
                    sel |= cur << k;
                }
                sel &= elig;
                carry_cont = last_cont >> 31;
                if (has) carry_dec = (ldec >> (31 - __clz(has))) & 1u;
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (((elig >> k) & 1u) && (mix64(R + (2ull * (uint64_t)(c0 + k) + 1ull) * GOLD) >> 32) < A.t_sel) sel |= 1u << k;
            }
            int32_t y[4];
            int64_t l[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                y[k] = x[k];
                l[k] = -100;
                if ((sel >> k) & 1u) {
                    const uint64_t v = mix64(R + (2ull * (uint64_t)(c0 + k) + 2ull) * GOLD);
                    const uint64_t u = v >> 32;
                    if (u < A.t_mask) y[k] = A.msk;
                    else if (u < A.t_mask_rand) y[k] = __ldg(&A.repl[((v & 0xFFFFFFFFull) * A.m) >> 32]);
                    l[k] = x[k];
                }
            }
            if (quad) {
                if (c0 < W) {
                    st_cs128(dst + c0, make_uint4((uint32_t)y[0], (uint32_t)y[1], (uint32_t)y[2], (uint32_t)y[3]));
                    st_cs128(lab + c0, make_uint4((uint32_t)l[0], (uint32_t)(l[0] >> 32), (uint32_t)l[1], (uint32_t)(l[1] >> 32)));
                    st_cs128(lab + c0 + 2, make_uint4((uint32_t)l[2], (uint32_t)(l[2] >> 32), (uint32_t)l[3], (uint32_t)(l[3] >> 32)));
                }
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (c0 + k < W) { __stcs(dst + c0 + k, y[k]); __stcs(reinterpret_cast<long long*>(lab + c0 + k), (long long)l[k]); }
            }
        }
    }
}

}  // namespace gzt
