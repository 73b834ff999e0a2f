// encode.cuh -- the fused row kernel: UTF-8 whitespace pre-split, word-cache lookup, framing,
// truncation, padding, attention_mask and token types, one launch per chunk of documents.
//
// Replaces, per document (file:line in /root/reference/genz_tokenize/tokenize.py):
//   :106      re.findall(r"\S+\n?", text)                 -> classify16 + word list
//   :108-114  per-word bpe() + split                      -> word-cache hit (bpe.cuh fills misses)
//   :120-121  piece -> id with <unk> fallback             -> stored in the cache slot
//   :126-135  [bos] + ids + [eos]                         -> positions 0 / 1+nA
//   :222-246  pair framing  <s> A </s> </s> B </s>
//   :141-146  __padding (pad / truncate to max_len)
//   :148-152  get_atttention_mask
//   :154-182  get_sequence_id + get_token_type, :252-258 token_type_ids
//
// Work decomposition.  A warp owns a TILE of D consecutive documents; their bytes are contiguous in the
// packed batch, so the warp streams them as one byte range in windows of 30x16 bytes (+2 look-ahead
// pieces): every lane classifies one 16-byte piece (LDG.128), word starts are compacted into a
// shared-memory word list, and then all 32 lanes look up one word each (key gather, hash, one 32-byte
// cache slot).  A segmented warp scan over (document, token count) gives every word its position in its
// row; the D rows are staged in shared memory and written with 16-byte streaming stores by the whole warp.
// Rows that met a word whose BPE is still pending are queued for a second pass (k_bpe_pending in between).
#pragma once
#include <cuda.h>   // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)

#include "device_common.cuh"

namespace gzt {

// ---- TMA write-out (MODE_FIXED) --------------------------------------------------------------------
// The [n, W] planes are written by the TMA unit instead of by store instructions: per tile of D rows the warp stages
// the first KR columns (the only ones that can hold real tokens) in shared memory in their final form and one lane
// issues 2-D tensor stores -- box [D x KR] from the staging area, box(es) [D x PB] for the pad columns from a
// block-wide constant buffer.  Rows that do not fit KR columns are queued for the generic second pass.
struct __align__(64) TmaPlanes {
    CUtensorMap ids_real, ids_pad, mask_real, mask_pad, tt_real, tt_pad;
    int32_t KR;   // staged columns per row (multiple of 16, <= W)
    int32_t PB;   // columns per pad box (multiple of 16; 0 = no pad columns)
};
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(m),
                 "r"((uint32_t)__cvta_generic_to_shared(smem)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__host__ __device__ __forceinline__ size_t r128(size_t x) { return (x + 127) & ~(size_t)127; }
// bytes of one staging buffer (ids int32 + mask [+ token types]) for D rows of KR columns, every plane 128-byte aligned
__host__ __device__ __forceinline__ size_t tma_stage_bytes(int D, int KR, bool pair) { return r128((size_t)D * KR * 4) + r128((size_t)D * KR) * (pair ? 2 : 1); }
// bytes of the block-wide constant pad buffers ([D x PB] pad ids + [D x PB] zero bytes)
__host__ __device__ __forceinline__ size_t tma_const_bytes(int D, int PB) { return r128((size_t)D * PB * 4) + r128((size_t)D * PB); }

enum RowMode { MODE_FIXED = 0, MODE_COUNT = 1, MODE_RAGGED = 2 };

struct Side {
    const uint8_t* bytes;   // 16-byte aligned, readable up to round_up(nbytes, 16) + 16
    const int64_t* off;     // [n+1]
    int64_t nbytes;
};

struct RowArgs {
    Side a, b;
    int32_t has_pair;
    int64_t n_rows;
    int32_t W;                 // FIXED: max_len
    int32_t D;                 // documents per tile (1..32)
    uint32_t flags;
    // FIXED outputs
    int32_t* ids; uint8_t* mask; int8_t* tt; int8_t* seq;
    int32_t* row_len; int32_t* seq_len; uint8_t* status;
    // COUNT output / RAGGED input: framed length per row, and what to keep
    int32_t* L;                // [n_rows] framed length (COUNT writes)
    const int64_t* row_off;    // RAGGED: start of each row in ids
    const int32_t* keep;       // RAGGED: number of framed tokens to copy
    // second pass over a row list
    const uint32_t* row_list;  // NULL = all rows
    uint32_t* redo_list;       // rows with cache misses (filled in pass 1)
    uint32_t* fix_list;        // rows whose token types need the generic kernel
    int8_t eos_i8;
    int8_t pad_i8;             // what __padding appends to token_type_ids: the pad id (tokenize.py:143 via :257), GENZTOK_PAD_MARK when it does not fit
    // return_offset=True (tokenize.py:105-117,225-234): words per side (COUNT writes), span table (RAGGED writes)
    int32_t* nwA; int32_t* nwB;
    const int64_t* span_off;   // [n_rows+1] first span entry of each row
    int32_t* spans;            // [entries][2]
    // offset_mapping (RAGGED, k_rows<..., OFFS>): [entries][2] byte (start, end) of each token in its document, aligned with ids.
    // Only the text's tokens are written: the caller zeroes the plane first, so framing, pads and a forced </s> read (0, 0).
    int32_t* offs;
    const uint16_t* plen;      // byte length of every piece in the word cache, at the index of its id in tok_arena (bpe.cuh)
};

static const int WIN_LANES = 30;            // pieces whose word starts a window handles; 2 more are look-ahead
static const int WLIST_CAP = WIN_LANES * 8; // at most 8 word starts per 16-byte piece
static const uint32_t F_DIRTY = 1u, F_SPECIAL = 2u, F_PADTOK = 4u;
static const uint32_t EM_LEN = 0xFFFFFu, EM_TRUNC = 1u << 20, EM_GENERIC = 1u << 21, EM_SKIP = 1u << 22, EM_SEQLONG = 1u << 23;

// get_sequence_id + get_token_type in closed form for one row (see seq_describe)
struct SeqDesc { int32_t p1, m, f1, f2, r1, r2, err; };

// per-warp shared memory (the D token rows follow for MODE_FIXED)
struct RaggedTile {            // MODE_COUNT / MODE_RAGGED only
    int64_t dout[32];          // row start in ids
    int64_t dsbase[32];        // spans: index of this side's first entry for the row
    int32_t dkeep[32];         // tokens to keep
    int32_t dshift[32];        // spans: added to a framed token position to get the reference's numbering
    int32_t dwrd[32];          // words met so far in this side
};
struct __align__(16) TileSmem {
    int32_t doff[34];          // document offsets of the tile for the side being walked, relative to the tile base (16-byte aligned)
    int32_t dpos[32];          // next token position per document
    int32_t dnA[32];           // tokens of side A per document
    uint32_t dflag[32];        // F_*
    uint32_t demit[32];        // FIXED: row length | EM_* for the write-out loop
    uint32_t bnd[32];          // document-start bits per piece of the current window
    uint32_t wlist[WLIST_CAP]; // word starts: position in window (9 bits) | bytes to first whitespace (7 bits, 0 = unknown) | document << 16
    union {                    // keeps 4 blocks of 8 warps per SM at max_len 128
        SeqDesc dsd[32];       // MODE_FIXED pairs: token-type description per row
        RaggedTile rg;
    };
};

// ---- byte classification -----------------------------------------------------------------------
// bit i of the result = high bit of byte i of x (x has only 0x80 bits set)
__device__ __forceinline__ uint32_t gather_msb(uint32_t x) { return (((x >> 7) * 0x00204081u) >> 21) & 0xFu; }

// ASCII whitespace of Python \s: 0x09-0x0D, 0x1C-0x20 (SURVEY.md A.1), SWAR over 4 bytes -> 0x80 flags
__device__ __forceinline__ uint32_t ascii_ws4(uint32_t w) {
    uint32_t lo = w & 0x7F7F7F7Fu;
    uint32_t ge09 = lo + 0x77777777u;   // bit7 set iff (b&0x7f) >= 0x09
    uint32_t ge0e = lo + 0x72727272u;   // >= 0x0E
    uint32_t ge1c = lo + 0x64646464u;   // >= 0x1C
    uint32_t ge21 = lo + 0x5F5F5F5Fu;   // >= 0x21
    return ((ge09 & ~ge0e) | (ge1c & ~ge21)) & ~w & 0x80808080u;
}
// bytes that can start a non-ASCII whitespace code point: 0xC2, 0xE1, 0xE2, 0xE3 -> 0x80 flags
__device__ __forceinline__ uint32_t ws_lead4(uint32_t w) {
    uint32_t lo = w & 0x7F7F7F7Fu;                // 0xC2 -> 0x42, 0xE1..0xE3 -> 0x61..0x63
    uint32_t ge42 = lo + 0x3E3E3E3Eu, ge43 = lo + 0x3D3D3D3Du, ge61 = lo + 0x1F1F1F1Fu, ge64 = lo + 0x1C1C1C1Cu;
    return ((ge42 & ~ge43) | (ge61 & ~ge64)) & w & 0x80808080u;
}
// bytes 0x80..0xA0: every second byte of a non-ASCII whitespace (80, 81, 85, 9A, A0) is one -> 0x80 flags.
// (Vietnamese letters are E1 BA/BB xx, C3 xx, C4 xx, C6 xx: their E1 leads fail this test on the next byte.)
__device__ __forceinline__ uint32_t ws_second4(uint32_t w) {
    uint32_t lo = w & 0x7F7F7F7Fu;
    return ~(lo + 0x5F5F5F5Fu) & w & 0x80808080u;   // high bit set and low 7 bits <= 0x20
}

__device__ __forceinline__ uint32_t byte_of(const uint4& w, int j) {
    uint32_t x = j < 8 ? (j < 4 ? w.x : w.y) : (j < 12 ? w.z : w.w);
    return (x >> ((j & 3) * 8)) & 0xFFu;
}

// Can any of these eight bytes end a word?  ASCII whitespace, or a lead of a multi-byte whitespace (C2, E1..E3) followed by a
// byte in 0x80..0xA0 -- the next byte of the last one is not known and counts as one.  (Vietnamese letters are E1 BA / E1 BB xx,
// C3 xx, C4 xx, C6 xx: they pass.)
__device__ __forceinline__ bool may_end_word8(uint64_t v) {
    const uint32_t x = (uint32_t)v, y = (uint32_t)(v >> 32);
    const uint32_t lx = ws_lead4(x), ly = ws_lead4(y), sx = ws_second4(x), sy = ws_second4(y);
    const uint32_t cand = (lx & __funnelshift_r(sx, sy, 8)) | (ly & ((sy >> 8) | 0x80000000u));
    return (ascii_ws4(x) | ascii_ws4(y) | cand) != 0u;
}

// Length (2 or 3) of the non-ASCII whitespace code point whose lead byte b0 sits at position p, else 0.
// The 19 non-ASCII members of \s: C2 85, C2 A0, E1 9A 80, E2 80 80..8A, E2 80 A8/A9/AF, E2 81 9F, E3 80 80.
// (positions are 32-bit offsets from the tile base `tb`)
__device__ __forceinline__ int multibyte_ws(uint32_t b0, const uint8_t* tb, int32_t p, int32_t e) {
    if (b0 == 0xC2) {
        if (p + 1 < e) { uint32_t b1 = tb[p + 1]; if (b1 == 0x85 || b1 == 0xA0) return 2; }
        return 0;
    }
    if (b0 < 0xE1 || b0 > 0xE3 || p + 2 >= e) return 0;
    uint32_t b1 = tb[p + 1];
    if (b0 == 0xE1) return (b1 == 0x9A && tb[p + 2] == 0x80) ? 3 : 0;
    if (b0 == 0xE3) return (b1 == 0x80 && tb[p + 2] == 0x80) ? 3 : 0;
    if (b1 == 0x80) { uint32_t b2 = tb[p + 2]; return ((b2 >= 0x80 && b2 <= 0x8A) || b2 == 0xA8 || b2 == 0xA9 || b2 == 0xAF) ? 3 : 0; }
    if (b1 == 0x81) return tb[p + 2] == 0x9F ? 3 : 0;
    return 0;
}

// index of the document that holds byte position p: largest k in [0, nd) with doff[k] <= p
__device__ __forceinline__ int doc_of(const int32_t* doff, int nd, int32_t p) {
    int lo = 0, hi = nd - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (doff[mid] <= p) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Whitespace bits of the 16 bytes at `a` (bits 0..15) plus spill into the next piece (bits 16,17).
// Bytes outside [S,E) count as whitespace; a multi-byte whitespace never straddles two documents.
__device__ __forceinline__ uint32_t classify16(const uint4& w, const uint8_t* tb, int32_t a, int32_t S, int32_t E, const int32_t* doff, int nd) {
    uint32_t inseg = 0xFFFFu;
    if (a < S) inseg &= 0xFFFFu << (S - a);
    if (a + 16 > E) inseg &= 0xFFFFu >> (a + 16 - E);
    uint32_t ws = gather_msb(ascii_ws4(w.x)) | (gather_msb(ascii_ws4(w.y)) << 4) | (gather_msb(ascii_ws4(w.z)) << 8) |
                  (gather_msb(ascii_ws4(w.w)) << 12);
    if ((w.x | w.y | w.z | w.w) & 0x80808080u) {
        uint32_t lead = gather_msb(ws_lead4(w.x)) | (gather_msb(ws_lead4(w.y)) << 4) | (gather_msb(ws_lead4(w.z)) << 8) |
                        (gather_msb(ws_lead4(w.w)) << 12);
        if (lead) {
            const uint32_t sec = gather_msb(ws_second4(w.x)) | (gather_msb(ws_second4(w.y)) << 4) | (gather_msb(ws_second4(w.z)) << 8) |
                                 (gather_msb(ws_second4(w.w)) << 12);
            lead &= inseg & ((sec >> 1) | 0x8000u);       // the byte after the lead must qualify (unknown for byte 15)
            while (lead) {
                const int j = __ffs(lead) - 1;
                lead &= lead - 1;
                const int l = multibyte_ws(byte_of(w, j), tb, a + j, E);
                if (l && a + j + l <= doff[doc_of(doff, nd, a + j) + 1]) ws |= ((1u << l) - 1) << j;
            }
        }
    }
    return (ws & 0x3FFFFu) | (~inseg & 0xFFFFu);
}

// First whitespace position at or after q (q is on a code point boundary or inside a non-ws one).
__device__ __noinline__ int32_t slow_word_end(const uint8_t* tb, int32_t q, int32_t e) {
    while (q < e) {
        // eight bytes a step while none of them is ASCII whitespace or can start a multi-byte one (long tokens: URLs, base64, ...)
        if (q + 8 <= e) {
            const uint64_t* a = reinterpret_cast<const uint64_t*>(reinterpret_cast<uintptr_t>(tb + q) & ~(uintptr_t)7);
            const uint64_t v = bytes8(a[0], a[1], (uint32_t)(reinterpret_cast<uintptr_t>(tb + q) & 7) * 8u);
            if (!may_end_word8(v)) { q += 8; continue; }
        }
        for (int k = 0; k < 8 && q < e; k++, q++) {
            const uint32_t b = tb[q];
            if (b <= 0x20) { if ((b >= 0x09 && b <= 0x0D) || b >= 0x1C) return q; }
            else if (b >= 0xC2 && multibyte_ws(b, tb, q, e)) return q;
        }
    }
    return e;
}

// ---- word -> cache slot --------------------------------------------------------------------------
// 24-byte zero-padded key of the word at [p, p+len), len <= 24, via aligned 16-byte loads.
__device__ __forceinline__ void load_key24(const uint8_t* tb, int32_t p, uint32_t len, uint64_t* k0, uint64_t* k1, uint64_t* k2) {
    const int32_t A = p & ~15;
    int sh = p & 15;
    const uint8_t* bytes = tb;
    const int need = sh + (int)len;
    uint4 v0 = ldg128(bytes + A);
    uint64_t q0 = ((uint64_t)v0.y << 32) | v0.x, q1 = ((uint64_t)v0.w << 32) | v0.z, q2 = 0, q3 = 0, q4 = 0;
    if (need > 16) {
        uint4 v1 = ldg128(bytes + A + 16);
        q2 = ((uint64_t)v1.y << 32) | v1.x;
        q3 = ((uint64_t)v1.w << 32) | v1.z;
        if (need > 32) {
            uint2 v2 = __ldg(reinterpret_cast<const uint2*>(bytes + A + 32));
            q4 = ((uint64_t)v2.y << 32) | v2.x;
        }
    }
    if (sh >= 8) { q0 = q1; q1 = q2; q2 = q3; q3 = q4; sh -= 8; }
    uint64_t r0 = q0, r1 = q1, r2 = q2;
    if (sh) {
        const int s8 = sh * 8;
        r0 = (q0 >> s8) | (q1 << (64 - s8));
        r1 = (q1 >> s8) | (q2 << (64 - s8));
        r2 = (q2 >> s8) | (q3 << (64 - s8));
    }
    if (len <= 8) { if (len < 8) r0 &= (1ULL << (len * 8)) - 1; r1 = 0; r2 = 0; }
    else if (len <= 16) { if (len < 16) r1 &= (1ULL << ((len - 8) * 8)) - 1; r2 = 0; }
    else if (len < 24) r2 &= (1ULL << ((len - 16) * 8)) - 1;
    *k0 = r0; *k1 = r1; *k2 = r2;
}

// The same key from two 16-byte pieces already in registers (word inside 32 bytes from its aligned start): lets the
// caller issue the piece loads before the word length is final.
__device__ __forceinline__ void key_from_pieces(const uint4& v0, const uint4& v1, int sh, uint32_t len, uint64_t* k0, uint64_t* k1, uint64_t* k2) {
    uint64_t q0 = ((uint64_t)v0.y << 32) | v0.x, q1 = ((uint64_t)v0.w << 32) | v0.z, q2 = ((uint64_t)v1.y << 32) | v1.x, q3 = ((uint64_t)v1.w << 32) | v1.z;
    if (sh >= 8) { q0 = q1; q1 = q2; q2 = q3; q3 = 0; sh -= 8; }
    uint64_t r0 = q0, r1 = q1, r2 = q2;
    if (sh) {
        const int s8 = sh * 8;
        r0 = (q0 >> s8) | (q1 << (64 - s8));
        r1 = (q1 >> s8) | (q2 << (64 - s8));
        r2 = (q2 >> s8) | (q3 << (64 - s8));
    }
    if (len <= 8) { if (len < 8) r0 &= (1ULL << (len * 8)) - 1; r1 = 0; r2 = 0; }
    else if (len <= 16) { if (len < 16) r1 &= (1ULL << ((len - 8) * 8)) - 1; r2 = 0; }
    else if (len < 24) r2 &= (1ULL << ((len - 16) * 8)) - 1;
    *k0 = r0; *k1 = r1; *k2 = r2;
}

// ... and from 40 bytes (two pieces and the next 8 bytes): any word of up to 24 bytes whatever its alignment
__device__ __forceinline__ void key_from_pieces40(const uint4& v0, const uint4& v1, const uint2& v2, int sh, uint32_t len, uint64_t* k0, uint64_t* k1, uint64_t* k2) {
    uint64_t q0 = ((uint64_t)v0.y << 32) | v0.x, q1 = ((uint64_t)v0.w << 32) | v0.z, q2 = ((uint64_t)v1.y << 32) | v1.x, q3 = ((uint64_t)v1.w << 32) | v1.z;
    uint64_t q4 = ((uint64_t)v2.y << 32) | v2.x;
    if (sh >= 8) { q0 = q1; q1 = q2; q2 = q3; q3 = q4; sh -= 8; }
    uint64_t r0 = q0, r1 = q1, r2 = q2;
    if (sh) {
        const int s8 = sh * 8;
        r0 = (q0 >> s8) | (q1 << (64 - s8));
        r1 = (q1 >> s8) | (q2 << (64 - s8));
        r2 = (q2 >> s8) | (q3 << (64 - s8));
    }
    if (len <= 8) { if (len < 8) r0 &= (1ULL << (len * 8)) - 1; r1 = 0; r2 = 0; }
    else if (len <= 16) { if (len < 16) r1 &= (1ULL << ((len - 8) * 8)) - 1; r2 = 0; }
    else if (len < 24) r2 &= (1ULL << ((len - 16) * 8)) - 1;
    *k0 = r0; *k1 = r1; *k2 = r2;
}

// the 24 bytes at byte offset sh of a 40-byte window, not yet zero padded
__device__ __forceinline__ void key_from_pieces40_nomask(const uint4& v0, const uint4& v1, const uint2& v2, int sh, uint64_t* k0, uint64_t* k1, uint64_t* k2) {
    uint64_t q0 = ((uint64_t)v0.y << 32) | v0.x, q1 = ((uint64_t)v0.w << 32) | v0.z, q2 = ((uint64_t)v1.y << 32) | v1.x, q3 = ((uint64_t)v1.w << 32) | v1.z;
    uint64_t q4 = ((uint64_t)v2.y << 32) | v2.x;
    if (sh >= 8) { q0 = q1; q1 = q2; q2 = q3; q3 = q4; sh -= 8; }
    uint64_t r0 = q0, r1 = q1, r2 = q2;
    if (sh) {
        const int s8 = sh * 8;
        r0 = (q0 >> s8) | (q1 << (64 - s8));
        r1 = (q1 >> s8) | (q2 << (64 - s8));
        r2 = (q2 >> s8) | (q3 << (64 - s8));
    }
    *k0 = r0; *k1 = r1; *k2 = r2;
}
// zero the key bytes from len on (len in 1..24), branch free on 32-bit halves
__device__ __forceinline__ void key_mask24(uint32_t len, uint64_t* k0, uint64_t* k1, uint64_t* k2) {
    auto m32 = [&](int i) -> uint32_t {
        const int nb = min(max((int)len - 4 * i, 0), 4);
        return nb ? (0xFFFFFFFFu >> (8 * (4 - nb))) : 0u;
    };
    *k0 &= ((uint64_t)m32(1) << 32) | m32(0);
    *k1 &= ((uint64_t)m32(3) << 32) | m32(2);
    *k2 &= ((uint64_t)m32(5) << 32) | m32(4);
}

// kp: a key in the arena (8-byte aligned, see the insert below), wptr: the word in the text (any alignment)
__device__ __noinline__ bool long_key_equal(const uint8_t* kp, const uint8_t* wptr, uint32_t len) {
    const uint64_t* k = reinterpret_cast<const uint64_t*>(kp);
    const uint64_t* q = reinterpret_cast<const uint64_t*>(reinterpret_cast<uintptr_t>(wptr) & ~(uintptr_t)7);
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(wptr) & 7) * 8u;
    uint64_t lo = q[0];
    uint32_t i = 0;
    for (; i + 8 <= len; i += 8) {
        const uint64_t hi = *++q;
        if (bytes8(lo, hi, sh) != *k++) return false;
        lo = hi;
    }
    if (i < len) {
        const uint64_t m = (1ULL << ((len - i) * 8)) - 1;
        if ((bytes8(lo, q[1], sh) ^ *k) & m) return false;
    }
    return true;
}

// Find the word in the cache or insert it (BPE pending).  Returns the slot's value word (VAL_*); for a word whose BPE has
// not run yet that is VAL_PENDING | index of its slot, so that a later kernel can fetch the value without looking the word
// up again.  With insert_ok == false (second passes) an absent word is reported as VAL_PENDING and nothing is written.
__device__ __forceinline__ uint32_t cache_find_or_insert(const WordCache& C, const uint8_t* wptr, uint32_t len, uint64_t k0, uint64_t k1,
                                                         uint64_t k2, uint32_t h, bool insert_ok) {
    uint32_t idx = h & C.mask;
    bool fresh = false;   // false: the first look at a slot may be served by L1
    for (uint32_t guard = 0;; guard++) {
        if (guard > (1u << 24)) { atomicAdd(&C.ctr[C_ERR], 1ULL); return VAL_PENDING; }   // never spin forever: report instead
        Slot* s = &C.slots[idx];
        const uint4 a = fresh ? ld_cg128(s) : *reinterpret_cast<const uint4*>(s);
        if (a.x == len) {
            const uint4 b = fresh ? ld_cg128(reinterpret_cast<const uint4*>(s) + 1) : *(reinterpret_cast<const uint4*>(s) + 1);
            const uint64_t s0 = ((uint64_t)a.w << 32) | a.z, s1 = ((uint64_t)b.y << 32) | b.x, s2 = ((uint64_t)b.w << 32) | b.z;
            bool eq;
            if (len <= KEY_INLINE) eq = (s0 == k0) & (s1 == k1) & (s2 == k2);
            else eq = s1 == k1 && long_key_equal(C.key_arena + s0, wptr, len);
            if (eq) return (a.y & VAL_KIND) == VAL_PENDING ? (VAL_PENDING | idx) : a.y;
        } else if (a.x == SLOT_EMPTY || a.x == SLOT_LOCKED) {
            if (!fresh) { fresh = true; continue; }          // L1 may be stale: look again in L2
            if (a.x == SLOT_LOCKED) continue;                // another thread is writing this slot
            if (!insert_ok) return VAL_PENDING;
            const uint32_t old = atomicCAS(&s->len, SLOT_EMPTY, SLOT_LOCKED);
            if (old != SLOT_EMPTY) continue;                 // lost the race: re-examine the same slot
            uint64_t v0 = k0;
            if (len > KEY_INLINE) {                      // the key goes to the arena, 8-byte aligned, eight bytes a step
                const uint64_t off = atomicAdd(&C.ctr[C_KEYS], (unsigned long long)((len + 7u) & ~7u));
                uint64_t* kp = reinterpret_cast<uint64_t*>(C.key_arena + off);
                const uint64_t* q = reinterpret_cast<const uint64_t*>(reinterpret_cast<uintptr_t>(wptr) & ~(uintptr_t)7);
                const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(wptr) & 7) * 8u;
                uint64_t lo = q[0];
                for (uint32_t i = 0; i < len; i += 8) { const uint64_t hi = *++q; *kp++ = bytes8(lo, hi, sh); lo = hi; }
                v0 = off;
            }
            s->val = VAL_PENDING; s->k0 = v0; s->k1 = k1; s->k2 = k2;
            __threadfence();
            st_release_u32(&s->len, len);
            atomicAdd(&C.ctr[C_SLOTS], 1ULL);
            const uint64_t pi = atomicAdd(&C.ctr[C_PENDING], 1ULL);
            if (pi < C.pending_cap) C.pending[pi] = idx;
            else atomicAdd(&C.ctr[C_ERR], 1ULL);
            return VAL_PENDING | idx;
        }
        idx = (idx + 1) & C.mask;
        fresh = false;
    }
}

// One probe of the word's home slot with ordinary (L1-cacheable) loads: the common case of a word already in the
// cache.  Returns false when the slot does not hold this word (then lookup_slow decides).
__device__ __forceinline__ bool cache_probe_fast(const WordCache& C, uint32_t len, uint64_t k0, uint64_t k1, uint64_t k2, uint32_t h, uint32_t* val) {
    const uint4* s = reinterpret_cast<const uint4*>(&C.slots[h & C.mask]);
    const uint4 a = s[0], b = s[1];
    const uint64_t s0 = ((uint64_t)a.w << 32) | a.z, s1 = ((uint64_t)b.y << 32) | b.x, s2 = ((uint64_t)b.w << 32) | b.z;
    *val = a.y;
    return (a.x == len) & (s0 == k0) & (s1 == k1) & (s2 == k2);
}

// Everything that is not the fast path: words whose end is not known from the window registers, long keys,
// probe chains, insertion.  Recomputes the word end from the bytes.  Out of line on purpose.
__device__ __noinline__ uint32_t lookup_slow(const WordCache& C, const uint8_t* tb, int32_t p, int32_t e_doc, int insert_ok) {
    int32_t end = slow_word_end(tb, p + 1, e_doc);
    if (end < e_doc && tb[end] == 0x0A) end++;                         // \S+\n?  (tokenize.py:106)
    const uint32_t len = (uint32_t)(end - p);
    uint64_t k0, k1, k2; uint32_t h;
    if (len <= KEY_INLINE) { load_key24(tb, p, len, &k0, &k1, &k2); h = hash_key24(k0, k1, k2, len); }
    else { k1 = hash_long(tb + p, len); k0 = 0; k2 = 0; h = fmix32((uint32_t)k1 ^ (uint32_t)(k1 >> 32)); }
    return cache_find_or_insert(C, tb + p, len, k0, k1, k2, h, insert_ok != 0);
}

// ---- token types for a pair row in closed form ---------------------------------------------------
// get_sequence_id + get_token_type (tokenize.py:154-182) evaluated on the known positions of
// </s> in a row without interior special ids (SURVEY.md A.4).  Generic rows go to k_post_rows.
__device__ __forceinline__ SeqDesc seq_describe(int32_t nA, int32_t L, int32_t W) {
    // eos positions of the final row T (length W): framed a, a+1, c=L-1 if they survive truncation, W-1 if truncated
    int32_t E0 = -1, E1 = -1, E2 = -1, E3 = -1; int ne = 0;
    const int32_t a = 1 + nA, c = L - 1;
    auto push = [&](int32_t v) { if (ne == 0) E0 = v; else if (ne == 1) E1 = v; else if (ne == 2) E2 = v; else E3 = v; ne++; };
    if (a <= W - 2) push(a);
    if (a + 1 <= W - 2) push(a + 1);
    if (c <= W - 2 && c > a + 1) push(c);
    if (L >= W) push(W - 1);
    SeqDesc d;
    d.p1 = E0;
    int32_t e = -1;
    if (ne > 1 && E1 >= d.p1 + 2 && E0 != E1 - 1) e = E1;
    else if (ne > 2 && E2 >= d.p1 + 2 && E1 != E2 - 1) e = E2;
    else if (ne > 3 && E3 >= d.p1 + 2 && E2 != E3 - 1) e = E3;
    d.m = e >= 0 ? e + 1 : W;
    int32_t N0 = -1, N1 = -1, N2 = -1, N3 = -1; int nn = 0;   // None positions after S[0]=0, S[m-1]=1
    auto pushn = [&](int32_t v) {
        if (v >= 0 && v < d.m && v != 0 && v != d.m - 1) { if (nn == 0) N0 = v; else if (nn == 1) N1 = v; else if (nn == 2) N2 = v; else N3 = v; nn++; }
    };
    pushn(E0); pushn(E1); pushn(E2); pushn(E3);
    d.f1 = N0; d.f2 = N1; d.r1 = N2; d.r2 = N3;
    d.err = nn < 2;
    return d;
}
__device__ __forceinline__ int32_t seq_value(const SeqDesc& d, int32_t i) {
    int32_t v = i < d.p1 ? 0 : 1;
    if (i == d.r1 || i == d.r2) v = -1;
    if (i == d.f1) v = 0;
    if (i == d.f2) v = 1;
    if (i == 0) v = 0;
    if (i == d.m - 1) v = 1;
    return v;
}
// token_type_ids / sequence_id bytes for positions i0..i0+3 of a fixed-width row
__device__ __forceinline__ void seq_words4(const SeqDesc& d, int32_t i0, int32_t W, int8_t eos_i8, int8_t pad_i8, uint32_t* ttw, uint32_t* sqw) {
    const int32_t hi = i0 + 3;
    auto in4 = [&](int32_t v) { return v >= i0 && v <= hi; };
    if (i0 >= d.m) { *ttw = 0x01010101u * (uint32_t)(uint8_t)pad_i8; *sqw = 0xFEFEFEFEu; return; }
    if (hi < d.m && !(in4(0) | in4(d.m - 1) | in4(d.f1) | in4(d.f2) | in4(d.r1) | in4(d.r2) | in4(d.p1))) {
        const uint32_t v = i0 < d.p1 ? 0u : 0x01010101u;
        *ttw = v; *sqw = v;
        return;
    }
    uint32_t t = 0, s = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int32_t i = i0 + k;
        const int32_t sv = i < d.m ? seq_value(d, i) : (int32_t)pad_i8;
        const int32_t tv = (d.m == W && i == W - 1) ? (int32_t)eos_i8 : sv;
        t |= ((uint32_t)tv & 0xFFu) << (8 * k);
        s |= ((uint32_t)(i < d.m ? sv : -2) & 0xFFu) << (8 * k);
    }
    *ttw = t; *sqw = s;
}

// ---- walking one side of a tile --------------------------------------------------------------------
// All 32 lanes call this.  ts->doff[0..nd] holds the side's document offsets relative to the tile base `tb`
// (16-byte aligned), ts->dpos[] the next token position of every row.  Tokens at positions < cap (<= limit) are
// delivered to rowbufs (FIXED) / ts->rg.dout (RAGGED); words of a row that has reached `limit` are not looked up.
// All byte positions are 32-bit offsets from tb.  OFFS (RAGGED only): also the byte span of every delivered token in its
// document into offs_out, beside the ids (a word's pieces tile it: their lengths are in plen, beside tok_arena).
template <int MODE, typename TokT, bool OFFS = false>
__device__ __forceinline__ void walk_side(const DevTables& T, const WordCache& C, const uint8_t* __restrict__ tb, TileSmem* ts, int nd,
                                          int lane, int32_t limit, int32_t cap, TokT* rowbufs, int32_t Wp, int32_t* ids_out, bool insert_ok, int32_t* spans, bool count_words,
                                          int32_t* offs_out = nullptr, const uint16_t* plen = nullptr) {
    static_assert(!OFFS || MODE == MODE_RAGGED, "offsets are written by the ragged pass");
    const int32_t S = ts->doff[0], E = ts->doff[nd];
    if (E <= S) return;
    // documents that are empty share their start with the next one: then the per-piece start bits cannot number
    // documents and every word finds its document by binary search instead
    const bool has_empty = __any_sync(FULL_MASK, lane < nd && ts->doff[lane + 1] == ts->doff[lane]);
    const int32_t spec_max = max(T.pad, max(T.bos, T.eos));
    int dbase = 0;                // documents that started before the current window
    const int32_t n_win = (E + 16 * WIN_LANES - 1) / (16 * WIN_LANES);
    uint32_t carry = 1u << 15;    // the byte before the tile is whitespace, nothing spills in
    for (int32_t w = 0; w < n_win; ++w) {
        const int32_t wbase = w * (16 * WIN_LANES);
        const int32_t a = wbase + lane * 16;
        // document starts inside this window -> bits per piece
        ts->bnd[lane] = 0;
        __syncwarp();
        if (lane + 1 < nd) {
            const uint32_t o = (uint32_t)(ts->doff[lane + 1] - wbase);
            if (o < 16u * 32u) atomicOr(&ts->bnd[o >> 4], 1u << (o & 15));
        }
        __syncwarp();
        uint32_t ws18 = 0xFFFFu;
        if (a < E) {
            const uint4 v = ldg128(tb + a);
            ws18 = classify16(v, tb, a, S, E, ts->doff, nd);
        }
        uint32_t prev = __shfl_up_sync(FULL_MASK, ws18, 1);
        if (lane == 0) prev = carry;
        carry = __shfl_sync(FULL_MASK, ws18, WIN_LANES - 1);
        const uint32_t nw = ~(ws18 | (prev >> 16)) & 0xFFFFu;
        const uint32_t b16 = ts->bnd[lane];
        uint32_t st = nw & (~((nw << 1) | ((~prev >> 15) & 1u)) | b16);
        if (lane >= WIN_LANES) st = 0;                      // look-ahead pieces: their words belong to the next window
        // non-whitespace bits of the following pieces: word ends without touching memory
        uint32_t win_lo = nw, win_hi = 0;
        {
            const uint32_t n1 = __shfl_down_sync(FULL_MASK, nw, 1), n2 = __shfl_down_sync(FULL_MASK, nw, 2), n3 = __shfl_down_sync(FULL_MASK, nw, 3);
            if (lane + 1 < 32) win_lo |= n1 << 16;
            if (lane + 2 < 32) win_hi = n2;
            if (lane + 3 < 32) win_hi |= n3 << 16;
        }
        const int known = 16 * ((32 - lane) < 4 ? (32 - lane) : 4);
        // ---- compact my word starts into the word list (and number the documents by counting start bits)
        const int cnt = __popc(st);
        int incl = cnt | (__popc(b16) << 16);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += t; }
        const int total = __shfl_sync(FULL_MASK, incl, 31) & 0xFFFF;
        const int dlane = dbase + (incl >> 16) - __popc(b16);           // document of the byte before my piece
        dbase += __shfl_sync(FULL_MASK, incl, WIN_LANES - 1) >> 16;
        int k = (incl & 0xFFFF) - cnt;
        while (st) {
            const int b = __ffs(st) - 1;
            st &= st - 1;
            // bytes from the word start to the first whitespace: first zero of the window above bit b
            const uint32_t zl = ~__funnelshift_r(win_lo, win_hi, b + 1);   // window bits b+1 .. b+32
            int run;
            if (zl) run = __ffs(zl);
            else { const uint32_t zh = ~(win_hi >> (b + 1)); run = 32 + __ffs(zh); }   // zh != 0: the shift brings in zeros
            if (b + run >= known) run = 0;                  // not decided inside the window registers
            const int doc = dlane + __popc(b16 & ((2u << b) - 1));
            ts->wlist[k++] = (uint32_t)((lane * 16 + b) | (run << 9) | (doc << 16));
        }
        __syncwarp();
        // ---- one word per lane
        for (int j0 = 0; j0 < total; j0 += 32) {
            const int j = j0 + lane;
            const bool has = j < total;
            int doc = 0x7FFF;
            uint32_t nt = 0, val = 0;
            bool pending = false;
            int32_t wpos = 0, wlen = 0;                                  // OFFS: the word's first byte (from tb) and its length
            if (has) {
                const uint32_t wl = ts->wlist[j];
                const int32_t p = wbase + (int32_t)(wl & 511u);
                doc = has_empty ? doc_of(ts->doff, nd, p) : (int)(wl >> 16);
                // a word of a row that is already full cannot matter (and need not be known): skip its lookup
                if (ts->dpos[doc] < limit) {
                    const int32_t run = (int32_t)((wl >> 9) & 127u);
                    const int32_t e_doc = ts->doff[doc + 1];
                    const int32_t end0 = min(p + run, e_doc);
                    // issue every load the fast path needs at once: the byte behind the word (\S+\n?, tokenize.py:106)
                    // and the one or two aligned pieces that hold the word and that byte
                    const int sh = p & 15;
                    const int32_t span = sh + (end0 - p) + 1;
                    const bool fast = run != 0 && (end0 - p) < (int32_t)KEY_INLINE && span <= 32;
                    uint32_t nlb = 0;
                    uint4 v0 = make_uint4(0, 0, 0, 0), v1 = make_uint4(0, 0, 0, 0);
                    if (end0 < e_doc) nlb = tb[end0];
                    if (fast) {
                        v0 = ldg128(tb + (p & ~15));
                        if (span > 16) v1 = ldg128(tb + (p & ~15) + 16);
                    }
                    const uint32_t len = (uint32_t)(end0 - p) + (nlb == 0x0A ? 1u : 0u);
                    bool hit = false;
                    if (fast) {
                        uint64_t k0, k1, k2;
                        key_from_pieces(v0, v1, sh, len, &k0, &k1, &k2);
                        hit = cache_probe_fast(C, len, k0, k1, k2, hash_key24(k0, k1, k2, len), &val);
                    }
                    if (!hit) val = lookup_slow(C, tb, p, e_doc, insert_ok ? 1 : 0);
                    if (OFFS) {
                        wpos = p;
                        if (hit) wlen = (int32_t)len;
                        else if ((val & VAL_KIND) == VAL_SINGLE) {            // (a list of pieces carries its lengths: only a single needs the end)
                            int32_t end = slow_word_end(tb, p + 1, e_doc);
                            if (end < e_doc && tb[end] == 0x0A) end++;          // \S+\n?  (tokenize.py:106)
                            wlen = end - p;
                        }
                    }
                    const uint32_t kind = val & VAL_KIND;
                    if (kind == VAL_SINGLE) nt = 1;
                    else if (kind == VAL_MULTI) nt = C.tok_arena[val & VAL_PAYLOAD];
                    else { pending = true; nt = 1; }                    // BPE not run yet: at least one token (positions stay lower bounds, so a row
                                                                        // still fills up and the walk can stop; the row is redone anyway)
                }
            }
            // position of my first token: inclusive count of nt over the lanes of my document up to me
            const int dprev = __shfl_up_sync(FULL_MASK, doc, 1);
            const uint32_t heads = __ballot_sync(FULL_MASK, lane == 0 || dprev != doc);
            const int seg0 = 31 - __clz(heads & ((2u << lane) - 1));   // first lane of my document in this batch
            uint32_t sc;
            if (__all_sync(FULL_MASK, nt <= 1)) {                        // the usual case: every word is one token
                const uint32_t ones = __ballot_sync(FULL_MASK, nt == 1);
                sc = __popc(ones & ((2u << lane) - 1) & ~((1u << seg0) - 1));
            } else {
                sc = nt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(FULL_MASK, sc, o);
                    if (lane - o >= seg0) sc += t;
                }
            }
            const bool seg_last = lane == 31 || ((heads >> (lane + 1)) & 1u);
            int32_t q = 0;
            if (has) q = ts->dpos[doc] + (int32_t)(sc - nt);
            // q is a lower bound of the word's position while earlier words are pending: if even that is past the
            // row's end the word is irrelevant, otherwise the row must be redone after k_bpe_pending (one lane per
            // document says so: with a cold cache every word is pending)
            {
                const bool dirty = pending && q < limit;
                const uint32_t dm = __ballot_sync(FULL_MASK, dirty);
                if (dirty && (__ffs(dm >> seg0) - 1 + seg0 == lane)) atomicOr(&ts->dflag[doc], F_DIRTY);
            }
            int wrank = 0, wbase_idx = 0;
            if (MODE != MODE_FIXED && count_words) {                     // word index inside the row (return_offset)
                wrank = lane - seg0;
                if (has) wbase_idx = ts->rg.dwrd[doc];
            }
            __syncwarp();
            if (has && seg_last) {
                ts->dpos[doc] = q + (int32_t)nt;
                if (MODE != MODE_FIXED && count_words) ts->rg.dwrd[doc] = wbase_idx + wrank + 1;
            }
            if (MODE == MODE_RAGGED && spans && has) {                   // (first, last) token of the word, tokenize.py:112-113
                int32_t* e = spans + 2 * (ts->rg.dsbase[doc] + 1 + wbase_idx + wrank);
                e[0] = q + ts->rg.dshift[doc];
                e[1] = q + (int32_t)nt - 1 + ts->rg.dshift[doc];
            }
            if (MODE != MODE_COUNT && has && nt && !pending) {
                TokT* dsts = nullptr; int32_t* dstg = nullptr; int32_t lim;
                if (MODE == MODE_FIXED) { dsts = rowbufs + (size_t)doc * Wp; lim = cap; }
                else { dstg = ids_out + ts->rg.dout[doc]; lim = ts->rg.dkeep[doc]; }
                uint32_t fl = 0;
                // OFFS: byte offsets are relative to the document's first byte (not the tile's or the chunk's)
                int2* dsto = nullptr;
                int32_t ob = 0;
                if (OFFS) { dsto = reinterpret_cast<int2*>(offs_out) + ts->rg.dout[doc]; ob = wpos - ts->doff[doc]; }
                if ((val & VAL_KIND) == VAL_SINGLE) {                     // (a list of one token is a word that is itself a special id: bpe.cuh)
                    const int32_t t = (int32_t)(val & VAL_PAYLOAD);
                    if (t <= spec_max) { if (t == T.eos || t == T.bos) fl |= F_SPECIAL; if (t == T.pad) fl |= F_PADTOK; }
                    if (q < lim) {
                        if (MODE == MODE_FIXED) dsts[q] = (TokT)t; else dstg[q] = t;
                        if (OFFS) dsto[q] = make_int2(ob, ob + wlen);
                    }
                } else {
                    const uint32_t* src = C.tok_arena + (val & VAL_PAYLOAD) + 1;
                    const uint16_t* pl = OFFS ? plen + (val & VAL_PAYLOAD) + 1 : nullptr;
                    for (uint32_t i = 0; i < nt && q < lim; i++, q++) {
                        const int32_t t = (int32_t)src[i];
                        if (t <= spec_max) { if (t == T.eos || t == T.bos) fl |= F_SPECIAL; if (t == T.pad) fl |= F_PADTOK; }
                        if (MODE == MODE_FIXED) dsts[q] = (TokT)t; else dstg[q] = t;
                        if (OFFS) { const int32_t oe = ob + (int32_t)pl[i]; dsto[q] = make_int2(ob, oe); ob = oe; }
                    }
                }
                if (fl) atomicOr(&ts->dflag[doc], fl);
            }
            __syncwarp();
        }
        if (MODE == MODE_FIXED) {                            // every row of the tile already full: stop reading (SURVEY.md 5.7)
            const int32_t pmin = __reduce_min_sync(FULL_MASK, lane < nd ? ts->dpos[lane] : 0x7FFFFFFF);
            if (pmin >= limit) break;
        }
    }
    __syncwarp();
}

// TokT: type of the rows staged in shared memory (uint16_t when every id fits: half the footprint, twice the blocks).
// TMA (MODE_FIXED, TokT = int32_t only): the planes are written by tensor stores from a final-form staging area (see TmaPlanes).
// OFFS (MODE_RAGGED): A.offs receives the tokens' byte offsets (see RowArgs); the other instantiations are unchanged by it.
template <int MODE, typename TokT, bool TMA, bool OFFS = false>
__global__ void __launch_bounds__(256, 4) k_rows(DevTables T, WordCache C, RowArgs A, const __grid_constant__ TmaPlanes M) {
    pdl_wait(); pdl_trigger();
    if (A.row_list && C.ctr[C_REDO] == 0) return;                   // second pass with nothing to redo (the usual case): before any set-up
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int32_t W = A.W, D = A.D;
    const int32_t KR = TMA ? M.KR : 0, PB = TMA ? M.PB : 0;
    const int32_t Wp = TMA ? KR : ((W + 3) & ~3);
    const bool tma_tt = TMA && A.has_pair && A.tt;
    const size_t stage_b = TMA ? tma_stage_bytes(D, KR, tma_tt) : 0;
    const size_t const_b = TMA && PB ? tma_const_bytes(D, PB) : 0;
    const size_t per_warp = TMA ? r128(sizeof(TileSmem)) + 2 * stage_b
                                : sizeof(TileSmem) + (MODE == MODE_FIXED ? (((size_t)D * Wp * sizeof(TokT) + 15) & ~(size_t)15) : 0);
    TileSmem* ts = reinterpret_cast<TileSmem*>(smem_raw + const_b + (size_t)wib * per_warp);
    uint8_t* const stage0 = reinterpret_cast<uint8_t*>(ts) + (TMA ? r128(sizeof(TileSmem)) : sizeof(TileSmem));
    TokT* rowbufs = reinterpret_cast<TokT*>(stage0);
    if (TMA && PB) {                                               // block-wide constants: pad ids, zero bytes
        const uint4 pad4 = make_uint4((uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad);
        uint4* cp = reinterpret_cast<uint4*>(smem_raw);
        const int n_pad = (int)(r128((size_t)D * PB * 4) >> 4), n_all = (int)(const_b >> 4);
        for (int i = threadIdx.x; i < n_all; i += blockDim.x) cp[i] = i < n_pad ? pad4 : make_uint4(0, 0, 0, 0);
        fence_proxy_async_smem();
        __syncthreads();
    }

    const uint32_t n_items = (uint32_t)(A.row_list ? C.ctr[C_REDO] : (unsigned long long)A.n_rows);   // rows per chunk < 2^31
    // a row list holds arbitrary rows: they are not contiguous in the text, so its tiles hold one document
    const uint32_t Dt = A.row_list ? 1u : (uint32_t)D;
    const uint32_t n_tiles = (n_items + Dt - 1) / Dt;
    const uint32_t n_warps = gridDim.x * (uint32_t)wpb;
    const int32_t limit = MODE == MODE_FIXED ? W - 1 : 0x7FFFFFFF;
    const int32_t cap = TMA ? min(limit, KR) : limit;            // positions that are staged
    const bool insert_ok = !A.row_list && MODE != MODE_RAGGED;   // second passes only look words up
    uint32_t tma_iter = 0;
    uint32_t tok_total = 0;
    for (uint32_t tile = blockIdx.x * (uint32_t)wpb + wib; tile < n_tiles; tile += n_warps) {
        const int64_t r0 = A.row_list ? (int64_t)A.row_list[tile] : (int64_t)(tile * Dt);
        const uint32_t left = n_items - tile * Dt;
        const int nd = (int)(Dt < left ? Dt : left);
        // ---- set up the tile
        // document offsets relative to the 16-byte aligned start of the tile's text (nd may be 32: 33 offsets)
        int64_t o64 = lane <= nd ? A.a.off[r0 + lane] : 0;
        const int64_t o32nd = nd == 32 ? A.a.off[r0 + 32] : 0;
        int64_t tbase = __shfl_sync(FULL_MASK, o64, 0) & ~(int64_t)15;
        if (lane <= nd) ts->doff[lane] = (int32_t)(o64 - tbase);
        if (nd == 32 && lane == 0) ts->doff[32] = (int32_t)(o32nd - tbase);
        const bool count_words = MODE != MODE_FIXED && ((MODE == MODE_COUNT && A.nwA) || (MODE == MODE_RAGGED && A.spans));
        if (TMA) {
            // this tile's staging buffer: free once the stores issued two tiles ago have read it; every id starts as pad
            rowbufs = reinterpret_cast<TokT*>(stage0 + (tma_iter & 1u) * stage_b);
            if (lane == 0) bulk_wait_read<1>();
            __syncwarp();
            const uint4 pad4 = make_uint4((uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad);
            for (int i = lane; i < D * (KR >> 2); i += 32) reinterpret_cast<uint4*>(rowbufs)[i] = pad4;
            __syncwarp();
        }
        if (lane < nd) {
            ts->dpos[lane] = 1;                                    // position 0 is <s> (tokenize.py:135)
            ts->dflag[lane] = 0;
            ts->rg.dwrd[lane] = 0;
            if (MODE == MODE_RAGGED && A.spans) { ts->rg.dsbase[lane] = A.span_off[r0 + lane]; ts->rg.dshift[lane] = 0; }
            if (MODE == MODE_FIXED) { if (cap > 0) rowbufs[(size_t)lane * Wp] = (TokT)T.bos; }
            if (MODE == MODE_RAGGED) {
                const int64_t ro = A.row_off[r0 + lane];
                const int32_t kp = A.keep[r0 + lane];
                ts->rg.dout[lane] = ro; ts->rg.dkeep[lane] = kp;
                if (kp > 0) A.ids[ro] = T.bos;
            }
        }
        __syncwarp();
        walk_side<MODE, TokT, OFFS>(T, C, A.a.bytes + tbase, ts, nd, lane, limit, cap, rowbufs, Wp, A.ids, insert_ok, A.spans, count_words, A.offs, A.plen);
        if (A.has_pair) {
            // ... </s> </s> B   (tokenize.py:237-239)
            if (lane < nd) {
                const int32_t pos = ts->dpos[lane];
                ts->dnA[lane] = pos - 1;
                if (MODE == MODE_FIXED) { TokT* rb = rowbufs + (size_t)lane * Wp; if (pos < cap) rb[pos] = (TokT)T.eos; if (pos + 1 < cap) rb[pos + 1] = (TokT)T.eos; }
                if (MODE == MODE_RAGGED) { int32_t* g = A.ids + ts->rg.dout[lane]; const int32_t kp = ts->rg.dkeep[lane]; if (pos < kp) g[pos] = T.eos; if (pos + 1 < kp) g[pos + 1] = T.eos; }
                ts->dpos[lane] = pos + 2;
                if (count_words) {
                    const int32_t nw = ts->rg.dwrd[lane];
                    if (MODE == MODE_COUNT) A.nwA[r0 + lane] = nw;
                    if (MODE == MODE_RAGGED) {
                        // offset = [(0,0)] + words + [(n+1,n+1)] for A (tokenize.py:105,116); B's entries follow, every
                        // value shifted by the NUMBER OF ENTRIES of A (tokenize.py:232-233)
                        int32_t* e = A.spans + 2 * ts->rg.dsbase[lane];
                        e[0] = 0; e[1] = 0;
                        e[2 * (nw + 1)] = pos; e[2 * (nw + 1) + 1] = pos;           // n+1 with n = pos-1 tokens
                        ts->rg.dsbase[lane] += nw + 2;
                        ts->rg.dshift[lane] = (nw + 2) - (pos + 2) + 1;             // B token at framed q -> (q - (pos+2) + 1) + (nw+2)
                        int32_t* f = A.spans + 2 * ts->rg.dsbase[lane];
                        f[0] = nw + 2; f[1] = nw + 2;
                    }
                    ts->rg.dwrd[lane] = 0;
                }
            }
            __syncwarp();
            o64 = lane <= nd ? A.b.off[r0 + lane] : 0;
            const int64_t p32nd = nd == 32 ? A.b.off[r0 + 32] : 0;
            tbase = __shfl_sync(FULL_MASK, o64, 0) & ~(int64_t)15;
            if (lane <= nd) ts->doff[lane] = (int32_t)(o64 - tbase);
            if (nd == 32 && lane == 0) ts->doff[32] = (int32_t)(p32nd - tbase);
            __syncwarp();
            walk_side<MODE, TokT, OFFS>(T, C, A.b.bytes + tbase, ts, nd, lane, limit, cap, rowbufs, Wp, A.ids, insert_ok, A.spans, count_words, A.offs, A.plen);
        }
        // ---- closing </s>, row bookkeeping (one lane per row)
        if (lane < nd) {
            const int32_t pos = ts->dpos[lane];
            const int32_t dL = pos + 1;                                // framed length (>= W when the walk stopped early)
            if (MODE == MODE_FIXED) { if (pos < cap) rowbufs[(size_t)lane * Wp + pos] = (TokT)T.eos; }
            if (MODE == MODE_RAGGED) { if (pos < ts->rg.dkeep[lane]) A.ids[ts->rg.dout[lane] + pos] = T.eos; }
            const uint32_t fl = ts->dflag[lane];
            SeqDesc sd;
            if (MODE == MODE_FIXED && A.has_pair) sd = seq_describe(ts->dnA[lane], dL, W);
            bool again = (fl & F_DIRTY) != 0;
            // TMA write-out: rows that need more than the KR staged columns, or a mask by value, take the generic second pass
            if (TMA) again |= (KR < W && (dL > KR || (A.has_pair && sd.m > KR))) || (fl & F_PADTOK);
            if (again) {
                if (!A.row_list) { const unsigned long long k = atomicAdd(&C.ctr[C_REDO], 1ULL); A.redo_list[k] = (uint32_t)(r0 + lane); }
                else atomicAdd(&C.ctr[C_ERR], 1ULL);   // cannot happen: every word of a redo row was inserted in pass 1
                if (MODE == MODE_FIXED) ts->demit[lane] = EM_SKIP;
            } else if (MODE == MODE_FIXED) {
                const int64_t dr = r0 + lane;
                const int32_t Lr = dL < W ? dL : W;
                ts->demit[lane] = (uint32_t)Lr | (dL >= W ? EM_TRUNC : 0u) | ((fl & F_PADTOK) ? EM_GENERIC : 0u);
                if (TMA && dL >= W) rowbufs[(size_t)lane * Wp + (W - 1)] = (TokT)T.eos;   // tokens[:max_len-1] + [eos] (KR == W here)
                if (A.row_len) A.row_len[dr] = Lr;
                if (!(fl & F_PADTOK)) tok_total += (uint32_t)Lr;       // rows with a pad id inside are counted from their mask
                if (A.has_pair) {
                    ts->dsd[lane] = sd;
                    if (sd.m > Lr) ts->demit[lane] |= EM_SEQLONG;       // token types run on over the pads (SURVEY.md A.4)
                    if (A.seq_len) A.seq_len[dr] = sd.m;
                    if (A.status) A.status[dr] = (uint8_t)sd.err;
                    if ((fl & F_SPECIAL) || !T.specials_distinct) { const unsigned long long k = atomicAdd(&C.ctr[C_FIX], 1ULL); A.fix_list[k] = (uint32_t)dr; }
                }
            }
            if (MODE == MODE_COUNT) A.L[r0 + lane] = dL;
            if (count_words) {
                const int32_t nw = ts->rg.dwrd[lane];
                if (MODE == MODE_COUNT) { if (A.has_pair) A.nwB[r0 + lane] = nw; else A.nwA[r0 + lane] = nw; }
                if (MODE == MODE_RAGGED) {
                    int32_t* e = A.spans + 2 * ts->rg.dsbase[lane];
                    if (!A.has_pair) { e[0] = 0; e[1] = 0; }
                    const int32_t tail = pos + ts->rg.dshift[lane];                    // (n+1) of this side in the reference's numbering
                    e[2 * (nw + 1)] = tail; e[2 * (nw + 1) + 1] = tail;
                }
            }
        }
        __syncwarp();
        if (MODE != MODE_FIXED) continue;
        if (TMA) {
            // ---- FIXED, TMA: mask (and token types) of the staged columns, then tensor stores issued by one lane
            uint8_t* const sm_mask = reinterpret_cast<uint8_t*>(rowbufs) + r128((size_t)D * KR * 4);
            uint8_t* const sm_tt = sm_mask + r128((size_t)D * KR);
            const int32_t qpr = KR >> 2;                                // quads per staged row
            for (int d = lane >> 2; d < D; d += 8) {
                const uint32_t em = d < nd ? ts->demit[d] : EM_SKIP;
                const int32_t Lr = (em & EM_SKIP) ? 0 : (int32_t)(em & EM_LEN);
                for (int32_t q = lane & 3; q < qpr; q += 4) {
                    const int32_t c = Lr - q * 4;
                    const uint32_t mk = c >= 4 ? 0x01010101u : (c <= 0 ? 0u : (0x01010101u & ((1u << (8 * c)) - 1)));
                    reinterpret_cast<uint32_t*>(sm_mask)[d * qpr + q] = mk;
                    if (tma_tt) {
                        uint32_t ttw = 0, sqw;
                        if (!(em & EM_SKIP)) seq_words4(ts->dsd[d], q * 4, W, A.eos_i8, A.pad_i8, &ttw, &sqw);
                        reinterpret_cast<uint32_t*>(sm_tt)[d * qpr + q] = ttw;
                    }
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                const int32_t r = (int32_t)r0;
                tma_store_2d(&M.ids_real, rowbufs, 0, r);
                tma_store_2d(&M.mask_real, sm_mask, 0, r);
                if (tma_tt) tma_store_2d(&M.tt_real, sm_tt, 0, r);
                if (PB) {
                    const uint8_t* zeros = smem_raw + r128((size_t)D * PB * 4);
                    for (int32_t c0 = KR; c0 < W; c0 += PB) {
                        tma_store_2d(&M.ids_pad, smem_raw, c0, r);
                        tma_store_2d(&M.mask_pad, zeros, c0, r);
                        if (tma_tt) tma_store_2d(&M.tt_pad, zeros, c0, r);
                    }
                }
                bulk_commit();
            }
            tma_iter++;
            continue;
        }
        // ---- FIXED: the warp writes its rows -----------------------------------------------------------
        if ((W & 15) == 0) {
            // Pass A: the quads that can hold real tokens (the first KQ of every row), 8 rows x 4 quads per step with
            // the select logic.  Pass B: everything behind them is padding: constant 16-byte stores, one row per step.
            uint32_t lr = 0;
            if (lane < nd) { const uint32_t em = ts->demit[lane]; lr = (em & EM_SKIP) ? 0u : (em & EM_LEN); }
            const int32_t KQ = (int32_t)(((__reduce_max_sync(FULL_MASK, lr) + 15u) >> 4) << 2);
            const size_t grow = (size_t)r0 * (size_t)W;
            for (int dg = 0; dg < nd; dg += 8) {
                const int d = dg + (lane >> 2);
                const uint32_t em = d < nd ? ts->demit[d] : EM_SKIP;
                for (int32_t qb = 0; qb < KQ; qb += 4) {
                    const int32_t i0 = (qb + (lane & 3)) * 4;
                    if (em & EM_SKIP) continue;
                    const bool lastq = i0 + 4 == W;
                    const int32_t c = (int32_t)(em & EM_LEN) - i0;      // real tokens from this quad on
                    const TokT* rb = rowbufs + (size_t)d * Wp + i0;
                    int4 v;
                    if (sizeof(TokT) == 4) v = *reinterpret_cast<const int4*>(rb);
                    else {
                        const uint2 h = *reinterpret_cast<const uint2*>(rb);
                        v = make_int4((int)(h.x & 0xFFFFu), (int)(h.x >> 16), (int)(h.y & 0xFFFFu), (int)(h.y >> 16));
                    }
                    uint32_t mk;
                    if (!(em & EM_GENERIC)) {
                        v.x = c > 0 ? v.x : T.pad; v.y = c > 1 ? v.y : T.pad; v.z = c > 2 ? v.z : T.pad; v.w = c > 3 ? v.w : T.pad;
                        if (lastq && (em & EM_TRUNC)) v.w = T.eos;
                        mk = c >= 4 ? 0x01010101u : (c <= 0 ? 0u : (0x01010101u & ((1u << (8 * c)) - 1)));
                    } else {                                            // a pad id inside the text: mask by value
                        int32_t x[4] = {v.x, v.y, v.z, v.w};
                        mk = 0;
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            x[k] = k < c ? ((lastq && k == 3 && (em & EM_TRUNC)) ? T.eos : x[k]) : T.pad;
                            mk |= (uint32_t)(x[k] != T.pad) << (8 * k);
                        }
                        v = make_int4(x[0], x[1], x[2], x[3]);
                        tok_total += (uint32_t)__popc(mk);
                    }
                    const size_t g = grow + (size_t)d * W + i0;
                    st_cs128(A.ids + g, make_uint4((uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w));
                    if (A.mask) st_cs32(A.mask + g, mk);
                    if (A.has_pair && (A.tt || A.seq)) {
                        uint32_t ttw, sqw;
                        seq_words4(ts->dsd[d], i0, W, A.eos_i8, A.pad_i8, &ttw, &sqw);
                        if (A.tt) st_cs32(A.tt + g, ttw);
                        if (A.seq) st_cs32(A.seq + g, sqw);
                    }
                }
            }
            const int32_t qn = (W >> 2) - KQ;                           // pad-only quads per row
            if (qn > 0) {
                const uint4 pad4 = make_uint4((uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad, (uint32_t)T.pad);
                const bool pairs_planes = A.has_pair && (A.tt || A.seq);
                // which rows to skip / which need computed token types, as warp-uniform bit masks (no per-row loads)
                uint32_t em_l = lane < nd ? ts->demit[lane] : EM_SKIP;
                const uint32_t skip_rows = __ballot_sync(FULL_MASK, (em_l & EM_SKIP) != 0);
                const uint32_t long_rows = __ballot_sync(FULL_MASK, (em_l & EM_SEQLONG) != 0);
                for (int32_t q = lane; q < qn; q += 32) {               // column block: usually a single pass
                    const int32_t i0 = (KQ + q) * 4;
                    int32_t* gi = A.ids + grow + i0;
                    uint8_t* gm = A.mask ? A.mask + grow + i0 : nullptr;
                    for (int d = 0; d < nd; d++, gi += W) {
                        if ((skip_rows >> d) & 1u) continue;
                        st_cs128(gi, pad4);
                        if (gm) st_cs32(gm + (size_t)d * W, 0u);
                        if (pairs_planes) {
                            uint32_t ttw = 0x01010101u * (uint32_t)(uint8_t)A.pad_i8, sqw = 0xFEFEFEFEu;
                            if ((long_rows >> d) & 1u) seq_words4(ts->dsd[d], i0, W, A.eos_i8, A.pad_i8, &ttw, &sqw);
                            const size_t g = grow + (size_t)d * W + i0;
                            if (A.tt) st_cs32(A.tt + g, ttw);
                            if (A.seq) st_cs32(A.seq + g, sqw);
                        }
                    }
                }
            }
        } else {
            for (int d = 0; d < nd; d++) {
                const uint32_t em = ts->demit[d];
                if (em & EM_SKIP) continue;
                const int64_t dr = r0 + d;
                const int32_t Lr = (int32_t)(em & EM_LEN);
                const bool trunc = (em & EM_TRUNC) != 0, generic_mask = (em & EM_GENERIC) != 0;
                const TokT* rb = rowbufs + (size_t)d * Wp;
                for (int32_t i = lane; i < W; i += 32) {
                    const int32_t t = i < Lr ? ((trunc && i == W - 1) ? T.eos : (int32_t)rb[i]) : T.pad;
                    A.ids[dr * W + i] = t;
                    if (generic_mask) tok_total += (uint32_t)(t != T.pad);
                    if (A.mask) A.mask[dr * W + i] = (uint8_t)(t != T.pad);
                    if (A.has_pair) {
                        const SeqDesc& sd = ts->dsd[d];
                        const int32_t sv = i < sd.m ? seq_value(sd, i) : (int32_t)A.pad_i8;
                        const int32_t tv = (sd.m == W && i == W - 1) ? (int32_t)A.eos_i8 : sv;
                        if (A.tt) A.tt[dr * W + i] = (int8_t)tv;
                        if (A.seq) A.seq[dr * W + i] = (int8_t)(i < sd.m ? sv : -2);
                    }
                }
            }
        }
        __syncwarp();
    }
    if (TMA) { if (lane == 0) bulk_wait<0>(); __syncwarp(); }   // shared memory must outlive the stores' reads
    if (MODE == MODE_FIXED) {
        tok_total = __reduce_add_sync(FULL_MASK, tok_total);   // < 2^32 per warp
        if (lane == 0 && tok_total) atomicAdd(&C.ctr[C_TOKENS], (unsigned long long)tok_total);
    }
}

}  // namespace gzt
