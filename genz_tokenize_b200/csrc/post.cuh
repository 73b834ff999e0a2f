// post.cuh -- generic per-row kernels: ragged-layout bookkeeping (row lengths, scan), and the
// value-driven attention_mask / sequence_id / token_type_ids pass used for ragged rows, for rows
// that contain special ids inside the text, and for the public helper methods.
//
//   k_row_lens     tokenize.py:141-146 (__padding) as lengths: what to keep, how long the row gets
//   k_scan_i64     exclusive scan -> row offsets (north_star step 5)
//   k_post_rows    tokenize.py:148-152 (mask), :163-182 (get_sequence_id), :154-161 (get_token_type),
//                  :256-258 (token_type_ids padding), evaluated on the actual id values
//   k_decode_*     tokenize.py:137-139 (decode) as a gather of precomputed per-id forms
#pragma once
#include "device_common.cuh"

namespace gzt {

struct LenArgs {
    const int32_t* L;      // framed length per row
    int64_t n_rows;
    int32_t has_max_len, max_len, padding, truncation;
    int32_t* keep;         // framed tokens copied
    int64_t* out_len;      // final row length
    uint8_t* tail;         // 0 none, 1 pad fill [keep, out_len), 2 eos at keep
    const int32_t* nwA; const int32_t* nwB;   // return_offset: words per side (NULL when not wanted)
    int64_t* span_cnt;     // entries of the row's offset list: (nwA + 2) [+ (nwB + 2)]
};

__global__ void k_row_lens(LenArgs A) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < A.n_rows; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t L = A.L[r];
        int64_t keep = L, out = L; uint8_t tail = 0;
        if (A.has_max_len && A.padding) {                       // tokenize.py:247
            if (L < (int64_t)A.max_len) { out = A.max_len; tail = 1; }          // :142-143
            else if (A.truncation) { keep = py_head(L, (int64_t)A.max_len - 1); out = keep + 1; tail = 2; }   // :144-145
        }
        A.keep[r] = (int32_t)keep; A.out_len[r] = out; A.tail[r] = tail;
        if (A.span_cnt) A.span_cnt[r] = (int64_t)A.nwA[r] + 2 + (A.nwB ? (int64_t)A.nwB[r] + 2 : 0);
    }
}

// out[0..n] = exclusive scan of in[0..n) (out[n] = total). One block.
__global__ void __launch_bounds__(1024) k_scan_i64(const int64_t* in, int64_t* out, int64_t n) {
    __shared__ int64_t warp_sums[32];
    __shared__ int64_t carry_s;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int64_t base = 0; base < n; base += 1024) {
        const int64_t i = base + threadIdx.x;
        int64_t v = i < n ? in[i] : 0, x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int64_t t = __shfl_up_sync(FULL_MASK, x, o); if (lane >= o) x += t; }
        if (lane == 31) warp_sums[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int64_t s = warp_sums[lane], y = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int64_t t = __shfl_up_sync(FULL_MASK, y, o); if (lane >= o) y += t; }
            warp_sums[lane] = y - s;
        }
        __syncthreads();
        const int64_t c = carry_s;
        const int64_t incl = c + warp_sums[wid] + x;
        if (i < n) out[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) out[n] = carry_s;
}

// Large inputs: tile-local scans + a scan of the tile totals + a fix-up pass.
static const int SCAN_TILE = 4096;          // elements per block (1024 threads x 4)
__global__ void __launch_bounds__(1024) k_scan_tiles(const int64_t* in, int64_t* out, int64_t* tile_sum, int64_t n) {
    __shared__ int64_t warp_sums[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * 4;
    int64_t v[4], s = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) { v[k] = base + k < n ? in[base + k] : 0; s += v[k]; }
    int64_t x = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int64_t t = __shfl_up_sync(FULL_MASK, x, o); if (lane >= o) x += t; }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int64_t w = warp_sums[lane], y = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int64_t t = __shfl_up_sync(FULL_MASK, y, o); if (lane >= o) y += t; }
        warp_sums[lane] = y - w;
        if (lane == 31) tile_sum[blockIdx.x] = y;
    }
    __syncthreads();
    int64_t run = warp_sums[wid] + x - s;       // exclusive prefix of this thread inside the tile
#pragma unroll
    for (int k = 0; k < 4; k++) { if (base + k < n) out[base + k] = run; run += v[k]; }
}
__global__ void __launch_bounds__(1024) k_scan_fix(int64_t* out, const int64_t* tile_excl, int64_t n, int64_t n_tiles) {
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * 4;
    const int64_t add = tile_excl[blockIdx.x];
#pragma unroll
    for (int k = 0; k < 4; k++) if (base + k < n) out[base + k] += add;
    if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = tile_excl[n_tiles];
}

struct PostArgs {
    int32_t* ids;              // flat
    const int64_t* row_off;    // NULL -> fixed layout, row r at r*W
    int32_t W;
    int64_t n_rows;
    const uint32_t* row_list;  // optional subset (count at ctr[C_FIX])
    const int32_t* keep;       // with tail: fill [keep, len) first
    const uint8_t* tail;
    uint8_t* mask;             // may be NULL
    int32_t has_pair;
    int8_t* tt; int8_t* seq;   // row-aligned planes, may be NULL
    int32_t* tt_len; int32_t* seq_len; uint8_t* status; int32_t* row_len;
    int32_t has_max_len, max_len, padding, truncation;
    int32_t raw_seq;           // 1: write get_sequence_id's result without get_token_type (helper API)
    int8_t eos_i8, pad_i8;
    unsigned long long* tokens_ctr;   // += sum(mask)
};

// KEEP2: a row whose status is already 2 (a pair truncation strategy that could not apply, written by k_window_rows<..., KEEP>)
// keeps it.
template <bool KEEP2 = false>
__global__ void __launch_bounds__(256) k_post_rows(DevTables T, PostArgs A, const unsigned long long* list_count) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t n_items = A.row_list ? *list_count : (uint64_t)A.n_rows;
    unsigned long long tok_total = 0;
    for (uint64_t it = warp; it < n_items; it += nwarps) {
        const int64_t r = A.row_list ? (int64_t)A.row_list[it] : (int64_t)it;
        const int64_t start = A.row_off ? A.row_off[r] : r * (int64_t)A.W;
        const int32_t n = A.row_off ? (int32_t)(A.row_off[r + 1] - start) : A.W;
        int32_t* Tk = A.ids + start;
        if (A.tail) {                                               // tokenize.py:143 / :145
            const int32_t kp = A.keep[r]; const uint8_t tl = A.tail[r];
            if (tl == 1) for (int32_t i = kp + lane; i < n; i += 32) Tk[i] = T.pad;
            else if (tl == 2 && lane == 0) Tk[kp] = T.eos;
            __syncwarp();
            if (A.row_len && lane == 0) A.row_len[r] = tl == 1 ? kp : n;
        }
        if (A.mask) {                                               // tokenize.py:148-152
            int32_t cnt = 0;
            for (int32_t i = lane; i < n; i += 32) { uint8_t on = Tk[i] != T.pad; A.mask[start + i] = on; cnt += on; }
            cnt = __reduce_add_sync(FULL_MASK, cnt);
            tok_total += (unsigned long long)cnt;
        }
        if (!A.has_pair) continue;
        // ---- get_sequence_id (tokenize.py:163-182)
        int32_t p1 = n;                                             // first </s>
        for (int32_t base = 0; base < n && p1 == n; base += 32) {
            const int32_t i = base + lane;
            const uint32_t m = __ballot_sync(FULL_MASK, i < n && Tk[i] == T.eos);
            if (m) p1 = base + __ffs(m) - 1;
        }
        int32_t e = -1;                                             // closing </s>: first i >= p1+2 with T[i]==eos and T[i-1]!=eos
        for (int32_t base = p1 + 2; base < n && e < 0; base += 32) {
            const int32_t i = base + lane;
            const uint32_t m = __ballot_sync(FULL_MASK, i < n && Tk[i] == T.eos && Tk[i - 1] != T.eos);
            if (m) e = base + __ffs(m) - 1;
        }
        const int32_t m_len = e >= 0 ? e + 1 : n;
        // ---- get_token_type (tokenize.py:154-161): S[0]=0, S[-1]=1, first two remaining None -> 0, 1
        int32_t f1 = -1, f2 = -1;
        if (!A.raw_seq) {
            for (int32_t base = 0; base < m_len && f2 < 0; base += 32) {
                const int32_t i = base + lane;
                bool none = false;
                if (i < m_len && i != 0 && i != m_len - 1) {
                    const int32_t t = Tk[i];
                    none = (i < p1 && t == T.bos) || i == p1 || (i > p1 && t == T.eos);
                }
                uint32_t m = __ballot_sync(FULL_MASK, none);
                if (m && f1 < 0) { f1 = base + __ffs(m) - 1; m &= m - 1; }
                if (m && f2 < 0) f2 = base + __ffs(m) - 1;
            }
        }
        const bool err = !A.raw_seq && (f2 < 0 || m_len == 0);
        // token_type_ids length (tokenize.py:256-258)
        int32_t tt_keep = m_len, tt_len = m_len; int tt_tail = 0;
        if (A.has_max_len && A.padding) {
            if (m_len < A.max_len) { tt_len = A.max_len; tt_tail = 1; }
            else if (A.truncation) { tt_keep = (int32_t)py_head(m_len, (int64_t)A.max_len - 1); tt_len = tt_keep + 1; tt_tail = 2; }
        }
        const int32_t hi = n;
        for (int32_t i = lane; i < hi; i += 32) {
            int32_t v = -2;
            if (i < m_len) {
                const int32_t t = Tk[i];
                const bool none = (i < p1 && t == T.bos) || i == p1 || (i > p1 && t == T.eos);
                v = none ? -1 : (i < p1 ? 0 : 1);
                if (!A.raw_seq) {
                    if (i == f1) v = 0;
                    if (i == f2) v = 1;
                    if (i == 0) v = 0;
                    if (i == m_len - 1) v = 1;
                }
            }
            if (A.seq) A.seq[start + i] = (int8_t)v;
            if (A.tt) {
                int32_t tv = i < tt_keep ? v : (tt_tail == 2 && i == tt_keep ? (int32_t)A.eos_i8 : (int32_t)A.pad_i8);
                if (i < tt_len) A.tt[start + i] = (int8_t)tv;
            }
        }
        if (lane == 0) {
            if (A.seq_len) A.seq_len[r] = m_len;
            if (A.tt_len) A.tt_len[r] = tt_len;
            if (A.status) A.status[r] = (KEEP2 && A.status[r] == 2) ? 2 : err ? 1 : 0;
        }
    }
    if (A.tokens_ctr && lane == 0 && tok_total) atomicAdd(A.tokens_ctr, tok_total);
}

// ---- decode (tokenize.py:137-139) ------------------------------------------------------------------
// What pass 1 leaves per row for pass 2.  A fixed-width row is mostly a run of pad ids behind the real ones: that run decodes to
// one short form repeated, so pass 2 writes it straight to global memory as 16-byte units of the periodic text and never reads
// those ids again.  n_lead < 0: no such run (the whole row goes through the staging buffer).
struct __align__(16) DecLead {
    int32_t n_lead;       // ids [0, n_lead) are staged; ids [n_lead, n-1) are all pad; id n-1 is the row's last piece
    int32_t lead_bytes;   // text bytes of ids [0, n_lead)
    uint32_t last_off;    // the last piece (its "nothing follows" form): offset into the form blob ...
    uint32_t last_len;    // ... and length
};

struct DecArgs {
    const int32_t* ids;
    const int64_t* ids_off;   // NULL -> n rows of `width`
    int32_t width;
    int64_t n_rows;
    int64_t* out_len;         // per row bytes (pass 1)
    const int64_t* out_off;   // per row start (pass 2)
    uint8_t* out;
    DecLead* lead;            // written by pass 1, read by pass 2
    unsigned long long* lead_sum;   // fixed-width pass 1: ids in front of the pad runs, summed (NULL: not wanted)
    unsigned long long* tile_ctr;   // fixed-width kernels: the next tile of 32 rows to hand out (zero at launch)
    long long capacity;             // write pass: bytes `out` can take; a batch that needs more is not written (<= 0: not checked)
    int32_t pick, wide_max;         // write pass, fixed-width rows: 0 = run; 1..3 = run only if the batch's average lead picks this kernel
};

__device__ __forceinline__ void dec_form(const DevTables& T, int32_t id, bool last, uint32_t* off, uint32_t* len) {
    const uint32_t k = (id >= 0 && id < T.n_ids) ? (uint32_t)id : (uint32_t)T.n_ids;   // decoder.get(i, unk_token)
    const uint32_t dsc = last ? T.last_desc[k] : T.mid_desc[k];
    *off = (dsc >> 8) * 8u;
    *len = dsc & 255u;
    if (*len == 255u) *len = last ? T.last_len[k] : T.mid_len[k];                       // very long vocab entry
}

static const int DEC_CAP = 2048;       // bytes staged per warp before a flush
static const int DEC_MAXFORM = 32;     // forms longer than this go straight to global memory
static const int DEC_MINRUN = 8;       // shortest trailing run of pad ids worth the direct path
static const int DEC_MAXRUNROW = 1 << 26;          // rows longer than this take the staged path only (32-bit byte counts, exact x % L)
static const int64_t DEC_MAXROW = 0x7FFFFF00ll;    // ids per row (32-bit positions inside a row)

// the form a pad id decodes to when another piece follows, if it can be written as a periodic text (1..8 bytes)
__device__ __forceinline__ uint32_t dec_pad_period(const DevTables& T, uint64_t* text) {
    uint32_t off, len;
    dec_form(T, T.pad, false, &off, &len);
    if (len < 1 || len > 8) return 0;
    *text = *reinterpret_cast<const uint64_t*>(T.form_blob + off);
    return len;
}
// x % L for L in 1..8 and x < 2^29 with M = ceil(2^32 / L): one multiply-high instead of a division
__device__ __forceinline__ uint32_t dec_mod(uint32_t x, uint32_t L, uint32_t M) { return L == 1u ? 0u : x - __umulhi(x, M) * L; }

// bytes of id's "another piece follows" form; counts the id as real when it is not pad and not the row's last id
#define DEC_MID(ID, I)                                                        \
    do {                                                                      \
        const int32_t _id = (ID);                                             \
        const uint32_t _k = min((uint32_t)_id, nid);                          \
        uint32_t _l = T.mid_desc[_k] & 255u;                                  \
        if (_l == 255u) _l = T.mid_len[_k];                                   \
        sum += _l;                                                            \
        if (_id != pad && (I) < lim) hi = (I);                                \
    } while (0)

// Pass 1: bytes per row, and the description of the row's trailing run of pad ids.  A lane reads four consecutive ids with one
// 16-byte load where the row is aligned; every id is taken as "followed by another piece" and the row's last id is corrected
// afterwards by all lanes alike.  One row per warp at a time does not keep enough bytes in flight for HBM (measured: 1.8 TB/s),
// so the first 256 ids of the warp's next row are loaded before this row is worked on, and the row after that is located.
__global__ void __launch_bounds__(256, 4) k_decode_len(DevTables T, DecArgs A) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const int32_t pad = T.pad;
    const uint32_t nid = (uint32_t)T.n_ids;                          // index of decoder.get's default (unk_token)
    uint64_t padP = 0;
    const uint32_t padL = dec_pad_period(T, &padP);
    auto locate = [&](uint64_t rr, const int32_t*& p, int& n) {      // row rr: its ids and how many
        p = A.ids; n = 0;
        if (rr < (uint64_t)A.n_rows) {
            const int64_t start = A.ids_off ? A.ids_off[rr] : (int64_t)rr * A.width;
            const int64_t n64 = A.ids_off ? A.ids_off[rr + 1] - start : A.width;
            n = (int)(n64 < DEC_MAXROW ? n64 : DEC_MAXROW);
            p = A.ids + start;
        }
    };
    auto first_ids = [&](const int32_t* p, int n, int4& a, int4& b) {   // ids [4 lane, +4) and [128 + 4 lane, +4) where they are whole vectors
        a = make_int4(0, 0, 0, 0); b = a;
        if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
            if (4 * lane + 3 < n) a = __ldcs(reinterpret_cast<const int4*>(p + 4 * lane));
            if (128 + 4 * lane + 3 < n) b = __ldcs(reinterpret_cast<const int4*>(p + 128 + 4 * lane));
        }
    };
    const int32_t *ids, *ids1, *ids2;
    int n, n1, n2;
    int4 va, vb, va1, vb1;
    locate(warp, ids, n);
    locate(warp + nwarps, ids1, n1);
    first_ids(ids, n, va, vb);
    for (uint64_t r = warp; r < (uint64_t)A.n_rows; r += nwarps) {
        locate(r + 2 * nwarps, ids2, n2);
        first_ids(ids1, n1, va1, vb1);
        const bool vec = (reinterpret_cast<uintptr_t>(ids) & 15) == 0;
        const int lim = n - 1;
        int64_t run = 0;
        int hi = -1;                                                 // highest index below n-1 whose id is not pad
        for (int base = 0; base < n; base += 128) {
            const int i0 = base + 4 * lane;
            uint32_t sum = 0;
            if (vec && i0 + 3 < n) {
                int4 v = va;
                if (base == 128) v = vb;
                if (base > 128) v = __ldcs(reinterpret_cast<const int4*>(ids + i0));
                DEC_MID(v.x, i0); DEC_MID(v.y, i0 + 1); DEC_MID(v.z, i0 + 2); DEC_MID(v.w, i0 + 3);
            } else {
#pragma unroll
                for (int k = 0; k < 4; k++) if (i0 + k < n) DEC_MID(ids[i0 + k], i0 + k);
            }
            run += __reduce_add_sync(FULL_MASK, sum);
        }
        uint32_t last_off = 0, last_len = 0;
        if (n > 0) {                                                 // the last id: "nothing follows" form instead
            const int32_t idl = ids[lim];
            const uint32_t k = min((uint32_t)idl, nid);
            uint32_t lm = T.mid_desc[k] & 255u;
            if (lm == 255u) lm = T.mid_len[k];
            dec_form(T, idl, true, &last_off, &last_len);
            run += (int64_t)last_len - (int64_t)lm;
        }
        if (A.lead) {
            hi = __reduce_max_sync(FULL_MASK, hi);
            if (lane == 0) {
                uint4 d = make_uint4(0xFFFFFFFFu, 0u, last_off, last_len);   // DecLead{n_lead = -1, lead_bytes, last_off, last_len}
                if (padL && n >= 2 && n < DEC_MAXRUNROW) {
                    const int cnt = n - 2 - hi;                      // pad ids in [hi + 1, n - 1)
                    const int64_t lead_bytes = run - last_len - (int64_t)cnt * padL;
                    if (cnt >= DEC_MINRUN && lead_bytes >= 0 && lead_bytes < (1ll << 31)) { d.x = (uint32_t)(hi + 1); d.y = (uint32_t)lead_bytes; }
                }
                *reinterpret_cast<uint4*>(A.lead + r) = d;
            }
        }
        if (lane == 0) A.out_len[r] = run;
        ids = ids1; n = n1; va = va1; vb = vb1;
        ids1 = ids2; n1 = n2;
    }
}

// Tiles of 32 rows are handed out by a counter rather than by a fixed stride: a grid of resident warps would otherwise end with
// some warps one tile short of the others (4.6 tiles per warp on a million rows).  A warp fetches the tile after this one ahead of time.
__device__ __forceinline__ uint64_t dec_next_tile(unsigned long long* ctr, int lane) {
    unsigned long long t = 0;
    if (lane == 0) t = atomicAdd(ctr, 1ull);
    return __shfl_sync(FULL_MASK, t, 0);
}
#ifndef DEC_LEN_MINB
#define DEC_LEN_MINB 6
#endif
// Pass 1 for fixed-width rows (no offsets, width a multiple of four, ids 16-byte aligned, width x longest form < 2^31): a warp
// takes 32 consecutive rows.
//  A. It reads them as a sequence of 128-id segments, four 16-byte loads in flight per lane, and only LOOKS FOR THE PAD RUN: the
//     highest index in front of the row's last id that does not hold the pad id (four compares per vector, one warp maximum per
//     row), and the last id.  Row j's result stays in lane j.
//  B. A lane per row then sums the form lengths of the ids in front of the run (read again: they were fetched a moment ago) --
//     the run itself is (number of pads) x (length of the pad form) -- and writes the row's byte count and description.
// Rows are mostly padding, so the table lookups, which bound the pass by instruction issue when done for every id (107 warp
// instructions per row of 128 ids), are done for a tenth of them.
template <int NSEG>   // 128-id segments per row when the width says so at compile time (1: up to 128 ids, 2: up to 256), 0: any
__global__ void __launch_bounds__(256, DEC_LEN_MINB) k_decode_len_fixed(DevTables T, DecArgs A) {
    const int lane = threadIdx.x & 31;
    const int32_t pad = T.pad;
    const uint32_t nid = (uint32_t)T.n_ids;
    uint64_t padP = 0;
    const uint32_t padL = dec_pad_period(T, &padP);
    uint32_t pad_len;                                                // bytes of the pad id's form when another piece follows
    { const uint32_t k = min((uint32_t)pad, nid); pad_len = T.mid_desc[k] & 255u; if (pad_len == 255u) pad_len = T.mid_len[k]; }
    const int W = A.width, lim = W - 1;
    const int nseg = NSEG ? NSEG : (W + 127) >> 7;
    const int own_lane = (lim & 127) >> 2;                           // the lane whose last vector ends with the row's last id
    const uint64_t n_tiles = ((uint64_t)A.n_rows + 31) >> 5;
    uint32_t lead_ids = 0;
    uint64_t tile_next = dec_next_tile(A.tile_ctr, lane);
    for (;;) {
        const uint64_t tile = tile_next;
        if (tile >= n_tiles) break;
        tile_next = dec_next_tile(A.tile_ctr, lane);
        const int64_t r0 = (int64_t)tile * 32;
        const int rows = (int)(A.n_rows - r0 < 32 ? A.n_rows - r0 : 32);
        const int32_t* p = A.ids + r0 * W;
        const int total = rows * nseg;
        int my_hi = -1; int32_t my_idl = 0;                          // lane j: row r0 + j
        int row = 0, seg = 0;                                        // the next segment to work on
        const int32_t* q = p + 4 * lane;                             // this lane's ids of that row
        int hi = -1; int32_t lastv = 0;
        for (int f0 = 0; f0 < total; f0 += 4) {
            int4 v[4];
            {
                const int32_t* lq = q; int ls = seg;
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int i0 = 128 * ls + 4 * lane;
                    v[u] = make_int4(pad, pad, pad, pad);
                    if (f0 + u < total && i0 < W) v[u] = *reinterpret_cast<const int4*>(lq + 128 * ls);
                    if (++ls == nseg) { ls = 0; lq += W; }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (f0 + u < total) {
                    const int i0 = 128 * seg + 4 * lane;
                    if (i0 < W) {
                        int h = -1;
                        if (v[u].x != pad) h = i0;
                        if (v[u].y != pad) h = i0 + 1;
                        if (v[u].z != pad) h = i0 + 2;
                        if (v[u].w != pad && i0 + 3 < lim) h = i0 + 3;       // (the row's last id is the w of its last vector: W is a multiple of four)
                        hi = max(hi, h);
                        lastv = v[u].w;
                    }
                    if (++seg == nseg) {                             // the row is complete
                        const int rhi = __reduce_max_sync(FULL_MASK, hi);
                        const int32_t idl = __shfl_sync(FULL_MASK, lastv, own_lane);
                        if (lane == row) { my_hi = rhi; my_idl = idl; }
                        hi = -1; seg = 0; row++; q += W;
                    }
                }
            }
        }
        if (lane < rows) {                                           // one row per lane
            const int32_t* rid = p + (int64_t)lane * W;
            const int n_lead = my_hi + 1;
            uint32_t sum = 0;
            int4 nxt = *reinterpret_cast<const int4*>(rid);
            for (int i0 = 0; i0 < n_lead; i0 += 4) {
                const int4 v4 = nxt;
                if (i0 + 4 < n_lead) nxt = *reinterpret_cast<const int4*>(rid + i0 + 4);
                const int32_t idv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    const uint32_t k = min((uint32_t)idv[t], nid);   // decoder.get(i, unk_token)
                    uint32_t l = T.mid_desc[k] & 255u;
                    if (l == 255u) l = T.mid_len[k];                 // very long vocab entry
                    if (i0 + t < n_lead) sum += l;
                }
            }
            uint32_t last_off, last_len;
            dec_form(T, my_idl, true, &last_off, &last_len);         // the last id takes its "nothing follows" form
            const int cnt = W - 1 - n_lead;                          // pad ids in [n_lead, W - 1)
            const uint32_t run = sum + (uint32_t)cnt * pad_len + last_len;
            uint4 d = make_uint4(0xFFFFFFFFu, 0u, last_off, last_len);
            if (padL && W >= 2 && W < DEC_MAXRUNROW && cnt >= DEC_MINRUN) { d.x = (uint32_t)n_lead; d.y = sum; }
            if (A.lead) *reinterpret_cast<uint4*>(A.lead + r0 + lane) = d;
            A.out_len[r0 + lane] = run;
            lead_ids += (int32_t)d.x >= 0 ? d.x : (uint32_t)W;
        }
    }
    // ids in front of the pad runs, summed over the batch: the host picks the write kernel by their average
    lead_ids = __reduce_add_sync(FULL_MASK, lead_ids);
    if (lane == 0 && A.lead_sum && lead_ids) atomicAdd(A.lead_sum, (unsigned long long)lead_ids);
}
#undef DEC_MID

// ---- pass 2 ----
// The write kernel for fixed-width rows by the batch's average lead (ids in front of the pad run; the length pass summed them):
// 1 = a lane per junction with 256 bytes (single sentences), 2 = the same with 512 bytes, 3 = the whole warp gathers 32 pieces at a time.
__host__ __device__ inline int dec_pick(unsigned long long lead_sum, long long n_rows, int wide_max) {
    if (lead_sum <= 14ull * (unsigned long long)n_rows) return 1;
    if (lead_sum <= (unsigned long long)wide_max * (unsigned long long)n_rows) return 2;
    return 3;
}
// Does this launch write?  Not when the text does not fit the caller's buffer (the host learns the size afterwards and calls
// again), and not when the host launched all three kernels for fixed-width rows and the batch picks another.
__device__ __forceinline__ bool dec_write_go(const DecArgs& A, int me) {
    if (A.capacity > 0 && A.out_off[A.n_rows] > A.capacity) return false;
    if (A.pick && dec_pick(*A.lead_sum, A.n_rows, A.wide_max) != me) return false;
    return true;
}
struct DecWarp {              // what a warp of the write pass keeps across rows
    uint8_t* ob;              // its staging buffer (DEC_CAP + 16 bytes of shared memory)
    const uint8_t* padtab;    // [8][16]: sixteen-byte units of the periodic pad text, one per phase
    uint64_t padP;            // the pad text itself (one period, little endian)
    uint32_t padL, padM, step;   // period, ceil(2^32 / period), 512 % period
    int lane;
};

// One row of the write pass.  `ld` is the row's DecLead (x < 0: no pad run); with a run, its text and the last piece behind it go
// straight to global memory as 16-byte units of the periodic pad text.  The ids before it are gathered into the warp's staging
// buffer, one batch of 32 ids at a time with the next batch's ids in flight (`id_first`: this lane's id of the first batch,
// loaded by the caller ahead of time), and written with aligned 16-byte stores (edges bytewise: neighbouring rows belong to
// other warps).
__device__ __forceinline__ void dec_write_row(const DevTables& T, uint8_t* out, const int32_t* ids, int n, int64_t g0, uint4 ld, int32_t id_first,
                                              const DecWarp& w) {
    const int lane = w.lane;
    uint8_t* ob = w.ob;
    int ne = n;                                             // ids that go through the staging buffer
    if ((int32_t)ld.x >= 0) {
        ne = (int32_t)ld.x;
        const uint32_t L = w.padL, total = (uint32_t)(n - 1 - ne) * L;
        uint8_t* pp = out + g0 + (int32_t)ld.y;                                     // the run's text starts here
        const uint32_t h = (0u - (uint32_t)reinterpret_cast<uintptr_t>(pp)) & 15u;  // bytes up to the next unit
        if (total >= h + 16u) {
            const uint32_t nu = (total - h) >> 4, tb = h + (nu << 4), t = total - tb;
            if ((uint32_t)lane < h) pp[lane] = w.padtab[lane];
            uint32_t ph = dec_mod(h + 16u * lane, L, w.padM);
            uint4* up = reinterpret_cast<uint4*>(pp + h) + lane;
#pragma unroll 1
            for (uint32_t u = lane; u < nu; u += 32, up += 32) {
                __stcs(up, *reinterpret_cast<const uint4*>(w.padtab + 16 * ph));
                ph += w.step; if (ph >= L) ph -= L;
            }
            if ((uint32_t)lane < t) pp[tb + lane] = w.padtab[16 * dec_mod(tb, L, w.padM) + lane];
        } else {
            for (uint32_t k = lane; k < total; k += 32) pp[k] = (uint8_t)(w.padP >> (8 * dec_mod(k, L, w.padM)));
        }
        const uint8_t* src = T.form_blob + ld.z;                                    // the last piece behind the run
#pragma unroll 1
        for (uint32_t k = lane; k < ld.w; k += 32) pp[total + k] = src[k];
    }
    uint8_t* gbase = out + (g0 & ~(int64_t)15);             // global address of ob[0]
    int lead = (int)(g0 & 15);                              // ob[0..lead) is not ours (previous row)
    int cur = lead;
    // flush ob[0..upto) (upto multiple of 16, or everything when last): aligned 16-byte stores, foreign/partial units bytewise
    auto flush = [&](int upto, bool last) {
        __syncwarp();
        const int nfull = last ? (cur & ~15) : upto;
        if (lead && nfull && lane >= lead && lane < 16) gbase[lane] = ob[lane];
#pragma unroll 1
        for (int u = (lane + (lead ? 1 : 0)) * 16; u < nfull; u += 512) *reinterpret_cast<uint4*>(gbase + u) = *reinterpret_cast<const uint4*>(ob + u);
        if (last) {
            const int rem = cur - nfull;                    // trailing partial unit
            if (lane < rem) { const int k = nfull + lane; if (!(nfull == 0 && k < lead)) gbase[k] = ob[k]; }
            return;
        }
        __syncwarp();
        const int rem = cur - nfull;
        uint8_t keep = 0;
        if (lane < rem) keep = ob[nfull + lane];
        __syncwarp();
        if (lane < rem) ob[lane] = keep;
        gbase += nfull; cur = rem; lead = 0;
        __syncwarp();
    };
    int32_t idn = id_first;
    for (int base = 0; base < ne; base += 32) {
        const int i = base + lane;
        const int32_t id = idn;
        if (base + 32 < ne) idn = i + 32 < ne ? ids[i + 32] : 0;           // the next batch's ids in flight
        uint32_t off = 0, len = 0;
        if (i < ne) dec_form(T, id, i == n - 1, &off, &len);
        const uint8_t* src = T.form_blob + off;
        uint32_t incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(FULL_MASK, incl, o); if (lane >= o) incl += t; }
        const uint32_t tot = __shfl_sync(FULL_MASK, incl, 31);
        const uint32_t maxlen = __reduce_max_sync(FULL_MASK, len);
        if (maxlen <= (uint32_t)DEC_MAXFORM) {
            if (cur + (int)tot > DEC_CAP) flush(cur & ~15, false);
            uint8_t* d = ob + cur + (incl - len);
            // Eight bytes per form and round, the rounds and the bytes inside a round from the top down, without a test per byte:
            // what a form writes behind its own end belongs to a later form of the batch, which writes it in a later
            // instruction (its byte index there is smaller), or to nobody (behind the batch: 7 bytes of slack, rewritten by
            // the next batch).
            for (int k0 = (int)((maxlen - 1u) & ~7u); k0 >= 0 && maxlen; k0 -= 8) {
                if ((uint32_t)k0 < len) {
                    const uint64_t v = *reinterpret_cast<const uint64_t*>(src + k0);   // forms are 8-byte aligned in the blob
                    const uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
                    volatile uint8_t* dk = d + k0;                  // volatile: the stores stay in this order
                    dk[7] = (uint8_t)(hi >> 24); dk[6] = (uint8_t)(hi >> 16); dk[5] = (uint8_t)(hi >> 8); dk[4] = (uint8_t)hi;
                    dk[3] = (uint8_t)(lo >> 24); dk[2] = (uint8_t)(lo >> 16); dk[1] = (uint8_t)(lo >> 8); dk[0] = (uint8_t)lo;
                }
                __syncwarp();
            }
            cur += (int)tot;
        } else {                                            // rare: a very long vocab entry -> write this batch directly
            if (cur > lead || lead) { /* push out what is staged so far, bytewise tail included */
                __syncwarp();
                for (int k = lead + lane; k < cur; k += 32) gbase[k] = ob[k];
            }
            uint8_t* d = gbase + cur + (incl - len);
            for (uint32_t k = 0; k < len; k++) d[k] = src[k];
            // restart the staging buffer at the new position
            const int64_t gpos = (gbase - out) + cur + (int64_t)tot;
            gbase = out + (gpos & ~(int64_t)15);
            lead = (int)(gpos & 15);
            cur = lead;
            __syncwarp();
        }
    }
    flush(0, true);
    __syncwarp();
}

__device__ __forceinline__ DecWarp dec_warp_setup(const DevTables& T, uint8_t (*stage)[DEC_CAP + 16], uint8_t (*padtab)[8][16]) {
    DecWarp w;
    w.lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    w.ob = stage[wib];
    w.padP = 0;
    w.padL = dec_pad_period(T, &w.padP);
    w.padM = w.padL > 1 ? (uint32_t)((0x100000000ull + w.padL - 1) / w.padL) : 0u;
    w.step = w.padL ? 512u % w.padL : 0u;
    if (w.lane < (int)w.padL) {
        int ph = w.lane;
        for (int k = 0; k < 16; k++) { padtab[wib][w.lane][k] = (uint8_t)(w.padP >> (8 * ph)); ph = ph + 1 == (int)w.padL ? 0 : ph + 1; }
    }
    w.padtab = &padtab[wib][0][0];
    __syncwarp();
    return w;
}

// Pass 2, any rows: a warp per row; the next row's offset and description are fetched while this row is written.
__global__ void __launch_bounds__(256, 4) k_decode_write(DevTables T, DecArgs A) {
    __shared__ __align__(16) uint8_t stage[8][DEC_CAP + 16];
    __shared__ __align__(16) uint8_t padtab[8][8][16];
    if (!dec_write_go(A, 0)) return;
    const DecWarp w = dec_warp_setup(T, stage, padtab);
    const int lane = w.lane;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const bool use_lead = A.lead != nullptr && w.padL != 0;
    int64_t g0 = 0;
    uint4 ldw = make_uint4(0xFFFFFFFFu, 0, 0, 0);
    if (warp < (uint64_t)A.n_rows) {
        g0 = A.out_off[warp];
        if (use_lead) ldw = *reinterpret_cast<const uint4*>(A.lead + warp);
    }
    for (uint64_t r = warp; r < (uint64_t)A.n_rows; r += nwarps) {
        const int64_t start = A.ids_off ? A.ids_off[r] : (int64_t)r * A.width;
        const int64_t n64 = A.ids_off ? A.ids_off[r + 1] - start : A.width;
        const int n = (int)(n64 < DEC_MAXROW ? n64 : DEC_MAXROW);
        const int32_t* ids = A.ids + start;
        const int64_t g0_cur = g0;
        const uint4 ld_cur = ldw;
        const int ne = (int32_t)ld_cur.x >= 0 ? (int32_t)ld_cur.x : n;
        const int32_t id_first = lane < ne ? ids[lane] : 0;
        {   // the next row of this warp
            const uint64_t rn = r + nwarps;
            if (rn < (uint64_t)A.n_rows) {
                g0 = A.out_off[rn];
                if (use_lead) ldw = *reinterpret_cast<const uint4*>(A.lead + rn);
            }
        }
        dec_write_row(T, A.out, ids, n, g0_cur, ld_cur, id_first, w);
    }
}

// Pass 2 for fixed-width rows with long leads (sentence pairs: ~20 pieces in front of the pad run): the pieces of a row are
// gathered by the whole warp, 32 at a time (dec_write_row).  A warp takes 32 consecutive rows, lane j reads row j's offset and description (coalesced, once
// per 32 rows) and hands them out by shuffle; the first ids of the next row are loaded before this row is written.
__global__ void __launch_bounds__(256, 5) k_decode_write_fixed_coop(DevTables T, DecArgs A) {
    __shared__ __align__(16) uint8_t stage[8][DEC_CAP + 16];
    __shared__ __align__(16) uint8_t padtab[8][8][16];
    if (!dec_write_go(A, 3)) return;
    const DecWarp w = dec_warp_setup(T, stage, padtab);
    const int lane = w.lane;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const bool use_lead = A.lead != nullptr && w.padL != 0;
    const int W = A.width;
    const uint64_t n_tiles = ((uint64_t)A.n_rows + 31) >> 5;
    for (uint64_t tile = warp; tile < n_tiles; tile += nwarps) {
        const int64_t r0 = (int64_t)tile * 32;
        const int rows = (int)(A.n_rows - r0 < 32 ? A.n_rows - r0 : 32);
        long long my_g0 = 0;
        uint4 my_ld = make_uint4(0xFFFFFFFFu, 0, 0, 0);
        if (lane < rows) {
            my_g0 = A.out_off[r0 + lane];
            if (use_lead) my_ld = *reinterpret_cast<const uint4*>(A.lead + r0 + lane);
        }
        const int32_t* ids = A.ids + r0 * W;
        int ne_next;
        { const int x = __shfl_sync(FULL_MASK, (int)my_ld.x, 0); ne_next = x >= 0 ? x : W; }
        int32_t id_next = lane < ne_next ? ids[lane] : 0;
        for (int j = 0; j < rows; j++, ids += W) {
            const int64_t g0 = __shfl_sync(FULL_MASK, my_g0, j);
            uint4 ld;
            ld.x = __shfl_sync(FULL_MASK, my_ld.x, j); ld.y = __shfl_sync(FULL_MASK, my_ld.y, j);
            ld.z = __shfl_sync(FULL_MASK, my_ld.z, j); ld.w = __shfl_sync(FULL_MASK, my_ld.w, j);
            const int32_t id_first = id_next;
            if (j + 1 < rows) {
                const int x = __shfl_sync(FULL_MASK, (int)my_ld.x, j + 1);
                ne_next = x >= 0 ? x : W;
                id_next = lane < ne_next ? ids[W + lane] : 0;
            }
            dec_write_row(T, A.out, ids, W, g0, ld, id_first, w);
        }
    }
}

// Pass 2 for fixed-width rows with short leads (single sentences: ~10 pieces in front of the pad run).  The text of consecutive
// rows is contiguous, so the output is cut at 16-byte boundaries inside the pad runs instead of at the rows: JUNCTION j is what
// lies between the last whole unit of row j-1's run and the first whole unit of row j's run -- the rest of run j-1, the last
// piece of row j-1, the pieces in front of row j's run (its "lead") and the first bytes of run j up to the next boundary.
// It begins and ends on a unit boundary, so every byte of the batch leaves in an aligned 16-byte store.
//  A. A LANE PER JUNCTION assembles it in shared memory from the two rows' descriptions (pass 1) -- the bytes go through a
//     64-bit accumulator and land as aligned 8-byte words; the 16-byte units of a junction are permuted by its lane number so
//     that neither these stores nor the unit loads of part B meet in one bank.
//  B. The WARP writes each junction and the whole units of the run behind it, a lane per unit.
//  Rows without a usable run, with a long lead or a long last piece are written whole by the general row routine afterwards
//  (a junction next to such a row starts or ends inside a unit: that unit goes bytewise).  There are n_rows + 1 junctions.
// STRIDE: bytes of shared memory per junction (16 or 32 units); the longest lead assembled there is STRIDE - 72:
// 15 (rest of the run before) + 24 (last piece) + lead + 15 (fill) <= STRIDE.
static const uint32_t DWJ_LASTMAX = 24;     // longest last piece
static const uint32_t DWJ_MINRUN = 48;      // shortest run (bytes): the two junctions around it must not meet
struct __align__(16) DwjInfo { long long base; uint32_t nrun; uint8_t nu, a, e, q0; };   // base: global offset of unit 0; a / e: first / last unit partial
__device__ __forceinline__ bool dwj_tail_ok(const uint4 ld, int W, uint32_t L, uint32_t* run_total) {
    const int32_t n_lead = (int32_t)ld.x;
    *run_total = n_lead >= 0 ? (uint32_t)(W - 1 - n_lead) * L : 0u;
    return n_lead >= 0 && *run_total >= DWJ_MINRUN && ld.w <= DWJ_LASTMAX;
}
template <int STRIDE, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB) k_decode_write_fixed(DevTables T, DecArgs A) {
    constexpr int DWJ_STRIDE = STRIDE, DWJ_LEADMAX = STRIDE - 72;
    constexpr uint32_t UMASK = STRIDE / 16 - 1;
    extern __shared__ __align__(16) uint8_t dwf_smem[];
    __shared__ __align__(16) uint8_t padtab[WARPS][8][16];
    __shared__ DwjInfo info[WARPS][32];
    if (!dec_write_go(A, STRIDE == 256 ? 1 : 2)) return;
    const int wib = threadIdx.x >> 5;
    uint8_t* const jbuf = dwf_smem + (size_t)wib * (32 * DWJ_STRIDE + 16);             // [32][STRIDE]; the general routine's staging buffer aliases it
    DecWarp w = dec_warp_setup(T, reinterpret_cast<uint8_t (*)[DEC_CAP + 16]>(dwf_smem), padtab);
    w.ob = jbuf;
    const int lane = w.lane;
    const int W = A.width;
    const uint32_t L = w.padL, nid = (uint32_t)T.n_ids;
    const uint64_t n_tiles = ((uint64_t)A.n_rows + 1 + 31) >> 5;
    const uint32_t sw2 = ((uint32_t)lane & UMASK) << 1;              // word wp of my junction lives in unit (wp >> 1) ^ (lane & UMASK): (wp ^ sw2) is its 8-byte word
    const uint32_t lane_ph = L ? dec_mod(16u * (uint32_t)lane, L, w.padM) : 0u;
    uint8_t* const mine = jbuf + lane * DWJ_STRIDE;
    uint64_t tile_next = dec_next_tile(A.tile_ctr, lane);
    for (;;) {
        const uint64_t tile = tile_next;
        if (tile >= n_tiles) break;
        tile_next = dec_next_tile(A.tile_ctr, lane);
        const int64_t j0 = (int64_t)tile * 32, jj = j0 + lane;
        // ---- A. my junction: between row jj - 1 and row jj
        const bool has_prev = jj >= 1 && jj <= A.n_rows, has_cur = jj < A.n_rows;
        uint4 ldp = make_uint4(0xFFFFFFFFu, 0, 0, 0), ldc = ldp;
        long long g0p = 0, g0c = 0;
        if (has_prev) { ldp = *reinterpret_cast<const uint4*>(A.lead + jj - 1); g0p = A.out_off[jj - 1]; }
        int4 first4 = make_int4(0, 0, 0, 0);
        if (has_cur) { ldc = *reinterpret_cast<const uint4*>(A.lead + jj); g0c = A.out_off[jj]; first4 = *reinterpret_cast<const int4*>(A.ids + jj * (int64_t)W); }
        if (tile_next < n_tiles) {   // what this warp's next tile will read first: into L2 while this one is worked on
            const int64_t jn = (int64_t)tile_next * 32 + lane;
            if (jn < A.n_rows) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(A.ids + jn * (int64_t)W));
                if ((lane & 7) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(A.lead + jn));
                if ((lane & 15) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(A.out_off + jn));
            }
        }
        uint32_t run_p = 0, run_c = 0;
        const bool pt = L != 0 && has_prev && dwj_tail_ok(ldp, W, L, &run_p);
        const bool cf = L != 0 && has_cur && dwj_tail_ok(ldc, W, L, &run_c) && ldc.y <= (uint32_t)DWJ_LEADMAX;
        const uint32_t slow_rows = __ballot_sync(FULL_MASK, has_cur && !cf);
        DwjInfo me; me.base = 0; me.nrun = 0; me.nu = 0; me.a = 0; me.e = 0; me.q0 = 0;
        if (pt || cf) {
            uint64_t acc = 0;
            uint32_t nb = 0, wp = 0;
            // v: eight bytes whose first `len` (1..8) are appended; the others must be zero (forms are zero-padded in the blob)
            auto append = [&](uint64_t v, uint32_t len) {
                const uint32_t sh = nb * 8u;
                acc |= v << sh;
                const uint32_t tot = nb + len;
                if (tot >= 8u) {
                    *reinterpret_cast<uint64_t*>(mine + ((wp ^ sw2) << 3)) = acc;
                    wp++;
                    acc = sh ? v >> (64u - sh) : 0ull;
                    nb = tot - 8u;
                } else nb = tot;
            };
            auto append_pad = [&](const uint8_t* p16, uint32_t cnt) {                   // cnt (1..15) bytes of the periodic text at p16
                const uint64_t lo = *reinterpret_cast<const uint64_t*>(p16);
                if (cnt >= 8u) {
                    append(lo, 8u);
                    if (cnt > 8u) append(*reinterpret_cast<const uint64_t*>(p16 + 8) & ~(~0ull << (8u * (cnt - 8u))), cnt - 8u);
                } else append(lo & ~(~0ull << (8u * cnt)), cnt);
            };
            if (pt) {
                const long long runstart = g0p + (long long)ldp.y, runend = runstart + (long long)run_p;
                me.base = runend & ~15ll;
                const uint32_t rt = (uint32_t)(runend & 15ll);
                if (rt) append_pad(w.padtab + 16u * dec_mod((uint32_t)(me.base - runstart), L, w.padM), rt);   // the rest of the run of row jj - 1
                const uint8_t* ls = T.form_blob + ldp.z;                                // its last piece (forms are padded to eight bytes in the blob)
                for (uint32_t b = 0; b < ldp.w; b += 8) append(*reinterpret_cast<const uint64_t*>(ls + b), min(8u, ldp.w - b));
            } else {
                me.base = g0c & ~15ll;
                me.a = (uint8_t)(g0c & 15ll);
                nb = me.a & 7u; wp = me.a >> 3;
            }
            if (cf) {
                const int32_t* rid = A.ids + jj * (int64_t)W;
                const int32_t n_lead = (int32_t)ldc.x;
                int4 nxt = first4;
                for (int32_t i0 = 0; i0 < n_lead; i0 += 4) {
                    const int4 v4 = nxt;
                    if (i0 + 4 < n_lead) nxt = *reinterpret_cast<const int4*>(rid + i0 + 4);   // (W is a multiple of 4 and the rows are 16-byte aligned)
                    const int32_t idv[4] = {v4.x, v4.y, v4.z, v4.w};
                    uint4 ff[4];
#pragma unroll
                    for (int t = 0; t < 4; t++) ff[t] = T.mid_fast[min((uint32_t)idv[t], nid)];                // decoder.get(i, unk_token)
#pragma unroll
                    for (int t = 0; t < 4; t++) {
                        if (i0 + t < n_lead) {
                            const uint32_t len = ff[t].w >> 24;
                            if (len <= 15u) {
                                if (len) append((uint64_t)ff[t].x | ((uint64_t)ff[t].y << 32), min(len, 8u));
                                if (len > 8u) append((uint64_t)ff[t].z | ((uint64_t)(ff[t].w & 0xFFFFFFu) << 32), len - 8u);
                            } else {                                                    // a longer piece: from the blob
                                const uint32_t dsc = T.mid_desc[min((uint32_t)idv[t], nid)], ln = dsc & 255u;   // (< 255: the lead is at most STRIDE - 72 bytes)
                                const uint8_t* src = T.form_blob + (dsc >> 8) * 8u;
                                for (uint32_t b = 0; b < ln; b += 8) append(*reinterpret_cast<const uint64_t*>(src + b), min(8u, ln - b));
                            }
                        }
                    }
                }
                const uint32_t pos = wp * 8u + nb, f = (0u - pos) & 15u;                // the run's first bytes, up to the next unit
                if (f) append_pad(w.padtab, f);
                me.q0 = (uint8_t)f;
            }
            const uint32_t pos_end = wp * 8u + nb;
            if (nb) *reinterpret_cast<uint64_t*>(mine + ((wp ^ sw2) << 3)) = acc;
            me.nu = (uint8_t)((pos_end + 15u) >> 4);
            me.e = (uint8_t)(pos_end & 15u);                                            // (0 behind a fill)
            me.q0 = (uint8_t)dec_mod((uint32_t)me.q0 + 512u * L - 16u * me.nu, L, w.padM);   // phase of the run's text at unit 0 of the junction
            if (cf) {
                const long long runend = g0c + (long long)ldc.y + (long long)run_c;
                me.nrun = (uint32_t)(((runend & ~15ll) - (me.base + (long long)pos_end)) >> 4);
            }
        }
        info[wib][lane] = me;
        const uint32_t todo = __ballot_sync(FULL_MASK, me.nu != 0 || me.nrun != 0);
        __syncwarp();
        // ---- B. the junctions and the runs behind them, one after the other, a lane per 16-byte unit
        for (uint32_t rest = todo; rest; rest &= rest - 1) {
            const int j = __ffs(rest) - 1;
            const DwjInfo ri = info[wib][j];
            const uint8_t* jb = jbuf + j * DWJ_STRIDE;
            const uint32_t nu = ri.nu, nt = nu + ri.nrun, sj = (uint32_t)j & UMASK;
            uint4* dst = reinterpret_cast<uint4*>(A.out + ri.base) + lane;
            uint32_t ph = (uint32_t)ri.q0 + lane_ph;                                     // unit u of the run's text: phase (q0 + 16 u) mod L
            if (ph >= L) ph -= L;
            if ((ri.a | ri.e) == 0) {                                                   // whole units only
                if ((uint32_t)lane < nt) __stcs(dst, *reinterpret_cast<const uint4*>((uint32_t)lane < nu ? jb + (((uint32_t)lane ^ sj) << 4) : w.padtab + 16u * ph));
            } else if ((uint32_t)lane < nt) {
                const uint32_t u = (uint32_t)lane;
                const uint8_t* su = u < nu ? jb + ((u ^ sj) << 4) : w.padtab + 16u * ph;
                const uint32_t lo = u == 0 ? ri.a : 0u, hi = (u == nu - 1 && ri.e) ? ri.e : 16u;
                if (lo == 0 && hi == 16u) __stcs(dst, *reinterpret_cast<const uint4*>(su));
                else for (uint32_t k = lo; k < hi; k++) reinterpret_cast<uint8_t*>(dst)[k] = su[k];
            }
#pragma unroll 1
            for (uint32_t u = (uint32_t)lane + 32u; u < nt; u += 32) {                   // (a junction has at most 32 units)
                ph += w.step; if (ph >= L) ph -= L;
                dst += 32;
                __stcs(dst, *reinterpret_cast<const uint4*>(w.padtab + 16u * ph));
            }
        }
        __syncwarp();
        // ---- the other rows: the general routine (its staging buffer is the junction buffer, free by now)
        for (uint32_t rest = slow_rows; rest; rest &= rest - 1) {
            const int j = __ffs(rest) - 1;
            const int64_t r = j0 + j;
            const long long g0 = A.out_off[r];
            const uint4 ld = A.lead ? *reinterpret_cast<const uint4*>(A.lead + r) : make_uint4(0xFFFFFFFFu, 0, 0, 0);
            const int32_t* ids = A.ids + r * (int64_t)W;
            const int ne = (int32_t)ld.x >= 0 ? (int32_t)ld.x : W;
            const int32_t id_first = lane < ne ? ids[lane] : 0;
            __syncwarp();
            dec_write_row(T, A.out, ids, W, g0, ld, id_first, w);
            __syncwarp();
        }
        __syncwarp();
    }
}

// ---- decode of ragged rows, one thread per id ------------------------------------------------------------
// Short ragged rows (about twenty ids each once the padding is trimmed) leave a warp per row mostly idle and pay its per-row
// arithmetic a million times.  Here every id is a thread: lengths per id, one scan over all ids, then each thread copies its
// form to where the scan says; neighbouring threads write neighbouring text.  Row offsets are the scan read at the row starts.
struct DecTokArgs {
    const int32_t* ids;       // ids of the whole batch; this chunk's ids are [base, base + n_ids)
    const int64_t* ids_off;   // n_rows + 1
    int64_t n_rows, base, n_ids;
    uint8_t* flag;            // n_ids: 1 = the id is the last of its row ("nothing follows" form)
    int64_t* len;             // n_ids: bytes per id
    const int64_t* pos;       // n_ids + 1: exclusive scan of len
    int64_t* out_off;         // n_rows + 1
    uint8_t* out;
    long long capacity;       // bytes `out` can take (<= 0: not checked); a batch that needs more is not written
};

__global__ void k_dectok_flags(DecTokArgs A) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= A.n_rows) return;
    const int64_t b = A.ids_off[r] - A.base, e = A.ids_off[r + 1] - A.base;
    if (e > b && b >= 0 && e <= A.n_ids) A.flag[e - 1] = 1;
}

__global__ void __launch_bounds__(256) k_dectok_len(DevTables T, DecTokArgs A) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n_ids) return;
    if (A.capacity > 0 && A.pos[A.n_ids] > A.capacity) return;
    uint32_t off, len;
    dec_form(T, A.ids[A.base + i], A.flag[i] != 0, &off, &len);
    A.len[i] = len;
}

__global__ void k_dectok_rowoff(DecTokArgs A) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > A.n_rows) return;
    int64_t b = A.ids_off[r] - A.base;
    b = b < 0 ? 0 : (b > A.n_ids ? A.n_ids : b);
    A.out_off[r] = A.pos[b];
}

__global__ void __launch_bounds__(256) k_dectok_write(DevTables T, DecTokArgs A) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.n_ids) return;
    if (A.capacity > 0 && A.pos[A.n_ids] > A.capacity) return;
    uint32_t off, len;
    dec_form(T, A.ids[A.base + i], A.flag[i] != 0, &off, &len);
    const uint8_t* src = T.form_blob + off;
    uint8_t* d = A.out + A.pos[i];
    for (uint32_t k0 = 0; k0 < len; k0 += 8) {                   // forms are 8-byte aligned in the blob: one load per 8 bytes
        const uint64_t v = *reinterpret_cast<const uint64_t*>(src + k0);
        const uint32_t nb = len - k0 < 8u ? len - k0 : 8u;
#pragma unroll
        for (uint32_t k = 0; k < 8; k++) if (k < nb) d[k0 + k] = (uint8_t)(v >> (8 * k));
    }
}

// get_atttention_mask helper on a flat id list
__global__ void k_mask_flat(const int32_t* ids, int64_t n, int32_t pad, uint8_t* out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = ids[i] != pad;
}

// Columns of a fixed-layout chunk that can differ from padding: max over rows of the row length and, for pairs, of the
// sequence-id length (token types run that far).  The host copies only those columns back (genztok.cu, encode_fixed_pipelined).
__global__ void __launch_bounds__(256) k_row_extent(const int32_t* row_len, const int32_t* seq_len, int64_t n, int32_t* out) {
    int32_t m = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        m = max(m, row_len[i]);
        if (seq_len) m = max(m, seq_len[i]);
    }
    m = __reduce_max_sync(FULL_MASK, m);
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}

// The first `wbytes` bytes (a multiple of 16) of every row of up to four [m, pitch] planes from device memory to mapped pinned
// host memory, 16 bytes a thread: the copy engine moves such 128-byte rows at a third of the link's rate, coalesced stores of an
// SM reach it.  (Runs on the copy-out stream beside the next chunk's kernels; a few blocks keep PCIe busy.)
struct CopyOutPlane { const uint8_t* src; uint8_t* dst; uint32_t pitch, wbytes; };
struct CopyOutArgs { CopyOutPlane p[4]; int32_t n_planes; int64_t m; };
__global__ void __launch_bounds__(256) k_copy_out(CopyOutArgs A) {
    for (int k = 0; k < A.n_planes; k++) {
        const CopyOutPlane P = A.p[k];
        const uint32_t upr = P.wbytes >> 4;                                   // 16-byte units per row
        const int64_t total = A.m * (int64_t)upr;
        for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
            const int64_t r = t / upr;
            const uint32_t u = (uint32_t)(t - r * upr);
            const size_t o = (size_t)r * P.pitch + (size_t)u * 16;
            *reinterpret_cast<uint4*>(P.dst + o) = __ldcs(reinterpret_cast<const uint4*>(P.src + o));
        }
    }
}

// ---- word cache housekeeping -------------------------------------------------------------------------
// Decide whether the cache can take the worst case of the next chunk; if not, schedule a reset.
__global__ void k_cache_guard(WordCache C, unsigned long long need_slots, unsigned long long need_keys, unsigned long long need_toks, int force) {
    pdl_wait(); pdl_trigger();
    unsigned long long* c = C.ctr;
    const unsigned long long cap = (unsigned long long)C.mask + 1;
    const bool reset = force || (c[C_SLOTS] + need_slots) * 2 > cap || c[C_KEYS] + need_keys > C.key_cap || c[C_TOKS] + need_toks > C.tok_cap;
    c[C_RESET] = reset;
    if (reset) { c[C_SLOTS] = 0; c[C_KEYS] = 0; c[C_TOKS] = 0; }
    c[C_PENDING] = 0; c[C_REDO] = 0; c[C_FIX] = 0; c[C_FLATFIX_A] = 0; c[C_FLATFIX_B] = 0; c[C_SCRATCH] = 0; c[C_TICKET] = 0; c[C_OVER32] = 0;
}
// ... and two optional word arrays to zero on the way (the document-start bitmaps of the byte-parallel pipeline)
__global__ void k_cache_clear(WordCache C, uint32_t* z0, uint64_t n0, uint32_t* z1, uint64_t n1) {
    pdl_wait(); pdl_trigger();
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = tid; i < n0; i += nth) z0[i] = 0u;
    for (uint64_t i = tid; i < n1; i += nth) z1[i] = 0u;
    if (!C.ctr[C_RESET]) return;
    uint4* p = reinterpret_cast<uint4*>(C.slots);
    const uint64_t n = ((uint64_t)C.mask + 1) * 2;
    const uint4 z = make_uint4(0, 0, 0, 0);
    for (uint64_t i = tid; i < n; i += nth) p[i] = z;
}
__global__ void k_reset_lists(WordCache C) { C.ctr[C_PENDING] = 0; C.ctr[C_REDO] = 0; C.ctr[C_FIX] = 0; C.ctr[C_FLATFIX_A] = 0; C.ctr[C_FLATFIX_B] = 0; C.ctr[C_TICKET] = 0; }

}  // namespace gzt
