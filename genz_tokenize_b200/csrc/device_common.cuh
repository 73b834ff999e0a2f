// device_common.cuh -- device-side tables, the word cache and small helpers shared by all kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "host_tables.hpp"

namespace gzt {

#define FULL_MASK 0xFFFFFFFFu

// ------------------------------------------------------------------------------------------------
// Model tables in HBM (built once per handle from vocab.txt / bpe.codes, < 4 MB, L2 resident)
// ------------------------------------------------------------------------------------------------
struct DevTables {
    const PairEntry* pair;   // (symL,symR) -> (rank, merged): tokenize.py:70-71 bpe_ranks.get(pair)
    uint32_t pair_mask;
    const CpEntry* cp;       // code point -> initial symbols "c" and "c</w>": tokenize.py:63-64
    uint32_t cp_mask;
    const int32_t* id_cont;  // symbol -> vocab id of S+"@@"  (tokenize.py:99,120)
    const int32_t* id_fin;   // symbol -> vocab id of S[:-4]  (tokenize.py:100,120)
    const uint32_t* sym_ncp; // symbol -> code points it spans
    int32_t pad, bos, eos, msk, unk;   // encoder[pad_token] ... looked up, not constant (SURVEY.md A.6)
    int32_t specials_distinct;         // bos, eos, pad pairwise different
    // decode forms (tokenize.py:137-139)
    const uint8_t* form_blob;
    const uint32_t *mid_off, *mid_len, *last_off, *last_len;
    const uint32_t *mid_desc, *last_desc;   // (offset/8) << 8 | min(len,255)
    const uint4* mid_fast;                  // a mid form of up to 15 bytes and, in byte 15, its length (255: longer, see mid_desc)
    int32_t n_ids;
};

// ------------------------------------------------------------------------------------------------
// Word cache: open-addressing hash keyed by the word's bytes, value = its token ids.
// One 32-byte slot = one L2 sector.  BPE runs once per distinct word (north_star step 2).
// ------------------------------------------------------------------------------------------------
struct __align__(32) Slot {
    uint32_t len;    // key length in bytes; SLOT_EMPTY / SLOT_LOCKED are states
    uint32_t val;    // VAL_PENDING | VAL_SINGLE|id | VAL_MULTI|offset into tok_arena (arena[off] = n, then n ids)
    uint64_t k0;     // len <= 24: key bytes 0..7 (zero padded); else offset into key_arena
    uint64_t k1;     // len <= 24: key bytes 8..15;              else 64-bit hash of the key
    uint64_t k2;     // len <= 24: key bytes 16..23;             else 0
};
static const uint32_t SLOT_EMPTY = 0u;
static const uint32_t SLOT_LOCKED = 0xFFFFFFFFu;
static const uint32_t KEY_INLINE = 24;
static const uint32_t VAL_PENDING = 0u, VAL_SINGLE = 1u << 30, VAL_MULTI = 2u << 30, VAL_KIND = 3u << 30, VAL_PAYLOAD = (1u << 30) - 1;

enum Counter { C_SLOTS = 0, C_KEYS = 1, C_TOKS = 2, C_PENDING = 3, C_REDO = 4, C_FIX = 5, C_RESET = 6, C_ERR = 7, C_TOKENS = 8, C_FLATFIX_A = 9, C_FLATFIX_B = 10, C_SCRATCH = 11, C_TICKET = 12, C_OVER32 = 13, C_COUNT = 16 };

struct WordCache {
    Slot* slots;
    uint32_t mask;            // capacity - 1
    uint8_t* key_arena;
    uint64_t key_cap;
    uint32_t* tok_arena;
    uint64_t tok_cap;
    uint32_t* pending;        // slot indices whose BPE has not run yet
    uint64_t pending_cap;
    unsigned long long* ctr;  // Counter[]
    uint32_t* rank_scratch;   // k_bpe_pending: pair ranks of the long words of this call (bpe.cuh)
    uint64_t rank_cap;
};

// Programmatic dependent launch: a kernel launched with the stream-serialization attribute may be scheduled while its
// predecessor drains; it must not touch the predecessor's results before pdl_wait().  pdl_trigger() lets the successor be scheduled.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg128(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
// A load that is really performed every time it is executed and is served by L2 (L1 may hold a stale copy of
// a cache slot another SM has just filled): used when re-examining a slot in the insert protocol.
__device__ __forceinline__ uint4 ld_cg128(const void* p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// streaming stores: outputs are written once and never re-read by this pipeline
__device__ __forceinline__ void st_cs128(void* p, uint4 v) { __stcs(reinterpret_cast<uint4*>(p), v); }
__device__ __forceinline__ void st_cs32(void* p, uint32_t v) { __stcs(reinterpret_cast<uint32_t*>(p), v); }

// splitmix64's finaliser and golden-ratio increment: the counter-based hashes of the synthetic workload, the plane digest
// (synth.cuh) and MLM masking (mlm.cuh); genz_tokenize_b200/workload.py::_mix64 is the same function on the host.
static const uint64_t GOLD = 0x9E3779B97F4A7C15ULL;
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ULL; x ^= x >> 27; x *= 0x94D049BB133111EBULL; x ^= x >> 31;
    return x;
}

__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return h;
}
// Hash of a <=24-byte zero-padded key held in three 64-bit registers: multiply-xor per 32-bit word, then a
// murmur finaliser.  (Every lookup verifies the full key, so quality only affects probe length.)
__device__ __forceinline__ uint32_t hash_key24(uint64_t k0, uint64_t k1, uint64_t k2, uint32_t len) {
    uint32_t h = len * 0x9E3779B1u;
    h += (uint32_t)k0 * 0xcc9e2d51u;
    h += (uint32_t)(k0 >> 32) * 0x1b873593u;
    h += (uint32_t)k1 * 0x85ebca6bu;
    h += (uint32_t)(k1 >> 32) * 0xc2b2ae35u;
    h += (uint32_t)k2 * 0x27d4eb2fu;
    h += (uint32_t)(k2 >> 32) * 0x165667b1u;
    h ^= h >> 15; h *= 0x2c1b3c6du; h ^= h >> 12; h *= 0x297a2d39u; h ^= h >> 15;
    return h;
}
// Bytes [p, p + 8) of a byte string at any alignment, out of aligned 8-byte loads: `lo` is the aligned word that holds p (the
// caller keeps it from the previous step), `hi` the next one.  Reads stay inside [p & ~7, (p & ~7) + 16): every text buffer
// is readable 16 bytes past its end (include/genztok.h), the key arena has the same slack.
__device__ __forceinline__ uint64_t bytes8(uint64_t lo, uint64_t hi, uint32_t sh) { return sh ? (lo >> sh) | (hi << (64u - sh)) : lo; }
// 64-bit hash of a long key, 8 bytes a step (one aligned load each)
__device__ __forceinline__ uint64_t hash_long(const uint8_t* p, uint32_t len) {
    const uint64_t* q = reinterpret_cast<const uint64_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)7);
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 7) * 8u;
    uint64_t h = 0xcbf29ce484222325ULL ^ len, lo = q[0];
    uint32_t i = 0;
    for (; i + 8 <= len; i += 8) {
        const uint64_t hi = *++q;
        h = (h ^ bytes8(lo, hi, sh)) * 0x9E3779B97F4A7C15ULL;
        h ^= h >> 29;
        lo = hi;
    }
    if (i < len) {
        const uint64_t v = bytes8(lo, q[1], sh) & ((1ULL << ((len - i) * 8)) - 1);
        h = (h ^ v) * 0x100000001b3ULL;
    }
    return h ^ (h >> 32);
}

// (symL,symR) -> rank, merged.  Returns 0xFFFFFFFF when the pair has no rank.
__device__ __forceinline__ uint32_t pair_rank(const DevTables& T, uint32_t l, uint32_t r, uint32_t* merged) {
    if (l == SYM_NONE || r == SYM_NONE) return 0xFFFFFFFFu;
    uint64_t x = ((uint64_t)l << 32) | r;
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    uint32_t i = (uint32_t)x & T.pair_mask;
    for (;;) {
        uint4 e = ldg128(&T.pair[i]);
        if (e.x == l && e.y == r) { *merged = e.w; return e.z; }
        if (e.x == SYM_NONE) return 0xFFFFFFFFu;
        i = (i + 1) & T.pair_mask;
    }
}
__device__ __forceinline__ void cp_symbols(const DevTables& T, uint32_t cp, uint32_t* mid, uint32_t* fin) {
    uint32_t i = ((cp * 0x9E3779B1u) ^ (cp >> 15)) & T.cp_mask;
    for (;;) {
        uint4 e = ldg128(&T.cp[i]);
        if (e.x == cp) { *mid = e.y; *fin = e.z; return; }
        if (e.x == SYM_NONE) { *mid = SYM_NONE; *fin = SYM_NONE; return; }
        i = (i + 1) & T.cp_mask;
    }
}

// Python tokens[:k] length
__host__ __device__ __forceinline__ int64_t py_head(int64_t len, int64_t k) {
    if (k < 0) { int64_t r = len + k; return r < 0 ? 0 : r; }
    return k < len ? k : len;
}

}  // namespace gzt
