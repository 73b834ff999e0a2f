// synth.cuh -- measurement plumbing, not part of the tokenizer: the synthetic workload of BASELINE.json configs[2]/[3]
// (100 M sentence pairs) produced on the device, and an order-independent digest of the output planes.
//
//   k_synth<false/true>  the counter-based generator of genz_tokenize_b200/workload.py::generate_hashed, same arithmetic
//                        bit for bit (tests/test_gpu_parity.py::test_synth_device_matches_host): a thread per document,
//                        lengths first, then -- after a scan -- the bytes.  Any range of documents can be produced
//                        independently, which is what lets N ranks shard one global batch by document.
//   k_plane_digest       sum over rows and 32-bit words of mix64((mix64(g * GOLD) + (plane << 32 | word index) * GOLD) ^ value)
//                        mod 2^64 over input_ids / attention_mask / token_type_ids, g = global row index: equal for any
//                        sharding and chunking of the same batch (SURVEY.md 8 d7: 1-GPU vs N-GPU full-output checksums).
#pragma once
#include "device_common.cuh"

namespace gzt {

struct SynthTables {
    const uint8_t* wblob; const uint32_t* wstart; const uint32_t* wlen; const uint32_t* cdf32; uint32_t nw;
    const uint8_t* eblob; const uint32_t* estart; const uint32_t* elen; uint32_t ne;
};
struct SynthArgs {
    uint64_t seed; int64_t doc0, n; int32_t side, lo, hi; uint32_t noise_thr;
    int64_t* len_out;            // lengths pass
    const int64_t* off;          // write pass: [n+1] byte offsets into `bytes`
    uint8_t* bytes;
};

static const uint64_t SY_K_LEN = 0xA5A5A5A5A5A5A5A5ULL, SY_K_NOISE = 0xC3C3C3C3C3C3C3C3ULL;
// first index with cdf32[i] > u (numpy searchsorted side='right'), clamped to nw - 1
__device__ __forceinline__ uint32_t synth_pick(const SynthTables& T, uint32_t u) {
    uint32_t lo = 0, hi = T.nw;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(&T.cdf32[mid]) <= u) lo = mid + 1; else hi = mid; }
    return lo < T.nw - 1 ? lo : T.nw - 1;
}

template <bool WRITE>
__global__ void __launch_bounds__(256) k_synth(SynthTables T, SynthArgs A) {
    const char alphabet[37] = "abcdefghijklmnopqrstuvwxyz0123456789";
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t d = (uint64_t)(A.doc0 + i);
        const uint64_t D = mix64(A.seed * GOLD + 2ULL * d + (uint64_t)A.side);
        const uint32_t k = (uint32_t)A.lo + (uint32_t)(((mix64(D ^ SY_K_LEN) >> 32) * (uint64_t)(A.hi - A.lo + 1)) >> 32);
        int64_t len = 0;
        uint8_t* out = WRITE ? A.bytes + A.off[i] : nullptr;
        auto put = [&](const uint8_t* src, uint32_t n) {
            if (WRITE) for (uint32_t t = 0; t < n; t++) out[len + t] = src[t];
            len += n;
        };
        for (uint32_t j = 0; j < k; j++) {
            const uint64_t R = mix64(D + (uint64_t)(j + 1) * GOLD);
            const uint32_t w = synth_pick(T, (uint32_t)(R >> 32));
            int kind = -1;
            uint64_t Q = 0;
            if ((uint32_t)R < A.noise_thr) { Q = mix64(R ^ SY_K_NOISE); kind = (int)(Q & 3ULL); }
            if (kind == 2) {                                      // a random string replaces the word
                const uint32_t n = 1u + (uint32_t)((Q >> 2) & 15ULL);
                const uint64_t h0 = mix64(Q + 1ULL), h1 = mix64(Q + 2ULL);
                for (uint32_t c = 0; c < n; c++) {
                    const uint32_t b = (uint32_t)(((c < 8 ? h0 : h1) >> (8 * (c & 7))) & 0xFFULL);
                    if (WRITE) out[len + c] = (uint8_t)alphabet[b % 36u];
                }
                len += n;
            } else {
                put(T.wblob + T.wstart[w], T.wlen[w]);
                if (kind >= 0) {
                    const uint32_t b = synth_pick(T, (uint32_t)(Q >> 32));
                    const uint32_t e = (uint32_t)(((Q >> 8) & 0xFFFFFFULL) % (uint64_t)T.ne);
                    if (kind == 0) put(T.wblob + T.wstart[b], T.wlen[b]);
                    else {
                        put(T.eblob + T.estart[e], T.elen[e]);
                        if (kind == 1) put(T.wblob + T.wstart[b], T.wlen[b]);
                    }
                }
            }
            if (j + 1 < k) { if (WRITE) out[len] = 0x20; len++; }
        }
        if (!WRITE) A.len_out[i] = len;
    }
}

struct DigestArgs {
    const uint32_t* ids; const uint32_t* mask; const uint32_t* tt;   // [n, W] words / [n, W/4] / [n, W/4] (tt may be NULL)
    int64_t n, row0; int32_t W;
    unsigned long long* acc;
};
__global__ void __launch_bounds__(256) k_plane_digest(DigestArgs A) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int32_t W = A.W, W4 = A.W >> 2;
    uint64_t sum = 0;
    for (int64_t r = warp; r < A.n; r += n_warps) {
        const uint64_t rk = mix64((uint64_t)(A.row0 + r) * GOLD);
        for (int32_t i = lane; i < W; i += 32) sum += mix64((rk + (uint64_t)i * GOLD) ^ (uint64_t)A.ids[r * W + i]);
        for (int32_t i = lane; i < W4; i += 32) {
            sum += mix64((rk + ((1ULL << 32) + (uint64_t)i) * GOLD) ^ (uint64_t)A.mask[r * W4 + i]);
            if (A.tt) sum += mix64((rk + ((2ULL << 32) + (uint64_t)i) * GOLD) ^ (uint64_t)A.tt[r * W4 + i]);
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(FULL_MASK, sum, o);
    if (lane == 0 && sum) atomicAdd(A.acc, (unsigned long long)sum);
}

}  // namespace gzt
