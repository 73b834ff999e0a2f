/*
 * genztok.h -- C ABI of libgenztok.so, the B200-native encode/decode engine behind the
 * `genz_tokenize.Tokenize` Python class.
 *
 * The reference (DVNghiem/genz-tokenize) has no FFI: its boundary is the public surface of
 * `class Tokenize` (genz_tokenize/tokenize.py:6-267).  Each entry point below names the reference
 * lines it replaces; the Python class in genz_tokenize_b200/tokenizer.py is a thin ctypes wrapper
 * over exactly these symbols (INTEGRATION.md shows the binding).
 *
 * Conventions
 *  - plain C types only; strings are (pointer, length) pairs, never NUL-terminated ('\0' is a
 *    legal word character, tokenize.py:106);
 *  - text is UTF-8 (the 'surrogatepass' form of a Python str); documents are packed back to back
 *    with int64 offsets[n+1];
 *  - every function returns 0 or a negative GENZTOK_E_* code and never throws; the message is
 *    available from genztok_last_error();
 *  - all tokenisation work runs in CUDA kernels on the handle's device(s).  There is no CPU
 *    fallback: a handle created with n_devices == 0 can only answer the table queries.
 */
#ifndef GENZTOK_H
#define GENZTOK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GENZTOK_OK 0
#define GENZTOK_E_INVALID (-1)  /* bad argument */
#define GENZTOK_E_IO (-2)       /* vocab / merges file cannot be opened (Python: FileNotFoundError) */
#define GENZTOK_E_UTF8 (-3)     /* vocab / merges file is not valid UTF-8 (Python: UnicodeDecodeError) */
#define GENZTOK_E_CUDA (-4)     /* CUDA runtime failure */
#define GENZTOK_E_NOMEM (-5)
#define GENZTOK_E_NODEVICE (-6) /* compute requested on a host-only handle */
#define GENZTOK_E_LIMIT (-7)    /* batch exceeds an engine limit (see DESIGN.md) */

/* `max_len` value meaning Python None (tokenize.py:187) */
#define GENZTOK_MAX_LEN_NONE INT32_MIN

/* `flags` of genztok_encode*: which optional planes to produce for sentence pairs */
#define GENZTOK_WANT_TOKEN_TYPE 1u  /* token_type_ids (tokenize.py:254-258) */
#define GENZTOK_WANT_SEQUENCE_ID 2u /* sequence_id    (tokenize.py:253-255) */
#define GENZTOK_WANT_SPANS 4u       /* return_offset=True word->token spans (tokenize.py:105-117,225-234) */
/* offset_mapping (HF tokenizers' return_offsets_mapping): per token, the int32 byte range [start, end) of the text it came from,
 * relative to the first byte of its own document (`text`, or `pair` for tokens of the second text).  The words are the matches
 * of \S+\n?; a word's BPE pieces tile it in order (an attached \n belongs to the last piece, an <unk> piece spans its code
 * point, a word that is a special token's text spans the word).  Tokens that do not come from the text -- <s>, </s> of the
 * framing, the </s> </s> between a pair's texts, pads, the </s> that truncation forces -- get (0, 0); every real token spans at
 * least one byte.  Asking for offsets changes no other output.  (Documents are limited to max_chunk_bytes <= 512 MiB, so every
 * byte offset fits an int32.) */
#define GENZTOK_WANT_OFFSETS 8u

/* Entries of the int8 planes */
#define GENZTOK_NONE (-1)      /* Python None */
#define GENZTOK_EOS_MARK (-3)  /* "the </s> id" when that id does not fit an int8 (tokenize.py:145 via :257) */
#define GENZTOK_PAD_MARK (-4)  /* "the <pad> id" in token_type_ids when that id does not fit an int8 (tokenize.py:143 via :257) */

typedef struct genztok genztok_t;

/* Result of an encode call.  All arrays are owned by the library (pinned host memory) until
 * genztok_free_encoded().  Layout: row r occupies [row_start(r), row_start(r) + row_width(r)) of
 * every flat plane, with row_start(r) = r*width when width > 0, else row_off[r].
 * sequence_id / token_type_ids are row-aligned: only their first seq_len[r] / tt_len[r] entries
 * are meaningful (the reference returns sequence_id unpadded, tokenize.py:253). */
typedef struct genztok_encoded {
    int64_t n;               /* rows */
    int64_t total;           /* entries in each flat plane */
    int32_t width;           /* > 0: fixed [n, width] layout (max_len >= 1, padding, truncation); 0: ragged */
    int32_t has_pair;
    int32_t *input_ids;      /* [total]  tokenize.py:250 */
    uint8_t *attention_mask; /* [total]  tokenize.py:148-152,251 */
    int64_t *row_off;        /* [n+1], NULL when width > 0 */
    int32_t *row_len;        /* [n] tokens in the row before padding (framing included) */
    int8_t *token_type_ids;  /* [total] or NULL */
    int8_t *sequence_id;     /* [total] or NULL */
    int32_t *tt_len;         /* [n] or NULL */
    int32_t *seq_len;        /* [n] or NULL */
    uint8_t *row_status;     /* [n] or NULL; 1 = the reference raises ValueError (tokenize.py:157-159) */
    int64_t *span_off;       /* [n+1] entries of `spans` per row, or NULL */
    int32_t *spans;          /* [span_off[n]][2] (first,last) token index pairs, or NULL */
    int64_t real_tokens;     /* sum over rows of attention_mask */
    void *_owner;            /* internal */
    int64_t d2h_bytes;       /* bytes this call copied from the device to the host (fixed layout: only the columns that can differ
                              * from padding travel; a recycled result buffer already holds the padding) */
    int32_t *offsets;        /* [total][2] (start, end) byte offsets with GENZTOK_WANT_OFFSETS, or NULL */
} genztok_encoded_t;

typedef struct genztok_text {
    int64_t n;
    int64_t total;    /* bytes */
    uint8_t *bytes;   /* UTF-8, rows back to back */
    int64_t *off;     /* [n+1] */
    void *_owner;
} genztok_text_t;

/* Device-resident planes for genztok_encode_device (fixed layout only); any pointer may be NULL
 * to skip that plane.  All are caller-allocated device memory on the handle's device. */
typedef struct genztok_dev_planes {
    int32_t *input_ids;      /* [n, max_len] */
    uint8_t *attention_mask; /* [n, max_len] */
    int8_t *token_type_ids;  /* [n, max_len] */
    int8_t *sequence_id;     /* [n, max_len], entries past seq_len[r] are GENZTOK_NONE - 1 */
    int32_t *row_len;        /* [n] */
    int32_t *seq_len;        /* [n] */
    uint8_t *row_status;     /* [n] */
    int32_t *offsets;        /* genztok_encode_windows_device: [n_windows, max_len, 2]; read only with GENZTOK_WANT_OFFSETS */
} genztok_dev_planes_t;

/* ---- lifetime: Tokenize.__init__ / Tokenize.fromFile (tokenize.py:7-42, 261-267) ------------ */
/* specials_utf8: pad,bos,eos,mask,unk strings (NULL or NULL entries = the reference defaults).
 * device_ids/n_devices: CUDA ordinals to run on; n_devices == 0 builds the tables only. */
int genztok_create(const char *vocab_path, const char *bpe_path, const char *const specials_utf8[5],
                   const int *device_ids, int n_devices, genztok_t **out);
void genztok_destroy(genztok_t *h);
const char *genztok_last_error(const genztok_t *h); /* h may be NULL: last create() failure */
const char *genztok_version(void);

/* ---- table queries (host side; valid on any handle) ----------------------------------------- */
int64_t genztok_vocab_size(const genztok_t *h);                 /* len(encoder), tokenize.py:59-60 */
int genztok_special_ids(const genztok_t *h, int32_t out[5]);    /* encoder[pad|bos|eos|mask|unk] */
/* encoder items in dict insertion order (tokenize.py:31-37,51) */
int64_t genztok_encoder_count(const genztok_t *h);
int genztok_encoder_entry(const genztok_t *h, int64_t i, const uint8_t **key, int64_t *key_len, int32_t *id);
/* encoder.get(key) -> id or -1 */
int32_t genztok_encoder_get(const genztok_t *h, const uint8_t *key, int64_t key_len);
/* decoder.get(id) (tokenize.py:40): 0 and *key=NULL when absent */
int genztok_decoder_get(const genztok_t *h, int64_t id, const uint8_t **key, int64_t *key_len);
/* merge lines as read by add_bpe_file (tokenize.py:53-57): line i has rank i */
int64_t genztok_merge_count(const genztok_t *h);
int genztok_merge_line(const genztok_t *h, int64_t i, const uint8_t **line, int64_t *line_len);
/* bpe_ranks.get((left,right)) -> rank or -1 */
int32_t genztok_rank_get(const genztok_t *h, const uint8_t *l, int64_t l_len, const uint8_t *r, int64_t r_len);

/* ---- encode: Tokenize.__call__ over a batch (tokenize.py:184-259) ---------------------------- */
/* Host buffers in, pinned host buffers out.  pair == NULL means pair_text=None for every row.
 * max_len == GENZTOK_MAX_LEN_NONE means None. */
int genztok_encode(genztok_t *h, const uint8_t *text, const int64_t *text_off, const uint8_t *pair,
                   const int64_t *pair_off, int64_t n, int32_t max_len, int padding, int truncation,
                   uint32_t flags, genztok_encoded_t *out);
void genztok_free_encoded(genztok_t *h, genztok_encoded_t *out);

/* Device buffers in, device buffers out, on `stream` (a cudaStream_t, NULL = the handle's own
 * stream) of device slot `dev` (index into device_ids).  Fixed layout only: requires
 * max_len >= 1, padding and truncation.  Asynchronous: returns after enqueueing.
 * GENZTOK_WANT_SPANS and GENZTOK_WANT_OFFSETS are rejected (GENZTOK_E_INVALID).  For offsets on the device use
 * genztok_encode_windows_device: window 0 of each document (rows d_win_off[:-1]) is its genztok_encode row. */
int genztok_encode_device(genztok_t *h, int dev, const uint8_t *d_text, const int64_t *d_text_off,
                          int64_t text_bytes, const uint8_t *d_pair, const int64_t *d_pair_off,
                          int64_t pair_bytes, int64_t n, int32_t max_len, uint32_t flags,
                          const genztok_dev_planes_t *planes, void *stream);

/* ---- long documents as overlapping windows (HF tokenizers' return_overflowing_tokens + stride) ---- */
/* T = encode(text)[1:-1] of L tokens (pairs: of the second text; A = the first text's, kept whole in every window).
 * Singles: C = max_len - 2; K = 1 if L <= C, else 1 + ceil((L - C) / (C - stride)); window k is
 * [bos] + T[k(C-stride) : k(C-stride)+C] + [eos].  Pairs: C = max_len - len(A) - 4, windows [bos] + A + [eos, eos] + B_k + [eos];
 * when C - stride < 1 the document yields one window, its genztok_encode(max_len) row (row_status included).  Every window is
 * then padded as tokenize.py:141-182,247-258 pad a row of max_len, so window 0 of a document equals its genztok_encode row.
 * Requires max_len >= 3 and 0 <= stride < max_len - 2. */
typedef struct genztok_windows {
    genztok_encoded_t enc;  /* fixed layout: enc.n = windows, enc.width = max_len */
    int64_t n_docs;
    int64_t *win_off;       /* [n_docs+1] first window of each document */
    int64_t *win_doc;       /* [enc.n] document of each window (overflow_to_sample_mapping) */
    int32_t *win_start;     /* [enc.n] index in T of the window's first content token */
} genztok_windows_t;
/* Host buffers in, pinned host buffers out (chunked and sharded across the handle's devices like genztok_encode).
 * flags: GENZTOK_WANT_TOKEN_TYPE / GENZTOK_WANT_SEQUENCE_ID for pairs, GENZTOK_WANT_OFFSETS (enc.offsets [K, max_len, 2]: a
 * token has the same offsets in every window that holds it). */
int genztok_encode_windows(genztok_t *h, const uint8_t *text, const int64_t *text_off, const uint8_t *pair,
                           const int64_t *pair_off, int64_t n, int32_t max_len, int32_t stride, uint32_t flags,
                           genztok_windows_t *out);
void genztok_free_windows(genztok_t *h, genztok_windows_t *out);
/* Device form, two steps like genztok_decode_device.  Step 1 (planes == NULL): tokenises, fills d_win_off[n+1] and returns
 * the number of windows in *n_windows (synchronises).  Step 2: writes the caller's [n_windows, max_len] planes (input_ids and
 * attention_mask required; row_len required; token types, seq_len, row_status for pairs) and d_win_doc / d_win_start [n_windows]
 * from what step 1 left in the handle; a step 2 for another batch (other pointers, n, max_len, stride, or GENZTOK_WANT_OFFSETS
 * other than in step 1) redoes step 1.  With GENZTOK_WANT_OFFSETS step 2 also fills planes->offsets [n_windows, max_len, 2].  Text
 * buffers 16-byte aligned, as for genztok_encode_device.  Step 2 does not synchronise. */
int genztok_encode_windows_device(genztok_t *h, int dev, const uint8_t *d_text, const int64_t *d_text_off, int64_t text_bytes,
                                  const uint8_t *d_pair, const int64_t *d_pair_off, int64_t pair_bytes, int64_t n, int32_t max_len,
                                  int32_t stride, uint32_t flags, int64_t *d_win_off, const genztok_dev_planes_t *planes,
                                  int64_t *d_win_doc, int32_t *d_win_start, int64_t *n_windows, void *stream);

/* ---- decode: Tokenize.decode over a batch (tokenize.py:137-139) ------------------------------ */
/* ids_off == NULL: n rows of `width` ids each.  Ids outside the decoder print the unk string. */
int genztok_decode(genztok_t *h, const int32_t *ids, const int64_t *ids_off, int64_t n, int32_t width,
                   genztok_text_t *out);
void genztok_free_text(genztok_t *h, genztok_text_t *out);
/* Device form: row byte lengths are produced first so that the caller can size `d_bytes`.
 * Step 1 (d_bytes == NULL): fills d_out_off[n+1] and returns the total in *total_bytes (synchronises; with ragged rows it
 * also reads the two ends of d_ids_off).  Step 2: writes the text; d_bytes 16-byte aligned.  Step 1 leaves a per-row (or
 * per-id) description in the handle for step 2 of the SAME batch (same pointers, n, width, on the same stream); a step 2
 * for another batch redoes it.  Rows hold fewer than 2^31 ids.  With several devices in the handle, genztok_decode shards
 * the rows across them. */
int genztok_decode_device(genztok_t *h, int dev, const int32_t *d_ids, const int64_t *d_ids_off, int64_t n,
                          int32_t width, int64_t *d_out_off, uint8_t *d_bytes, int64_t *total_bytes, void *stream);
/* Both steps at once into a buffer the caller already has (a ring reused across streamed batches): offsets into
 * d_out_off[n+1], text into d_bytes[capacity], no host read in between -- the kernels themselves check that the text fits
 * and write nothing when it does not.  total_bytes == NULL: the call does not synchronise (read d_out_off[n] later);
 * otherwise *total_bytes = bytes needed, after a synchronisation at the END of the call; when it exceeds `capacity`
 * call again with a larger buffer.  Same rows, same text as genztok_decode_device (tokenize.py:137-139). */
int genztok_decode_device_into(genztok_t *h, int dev, const int32_t *d_ids, const int64_t *d_ids_off, int64_t n,
                               int32_t width, int64_t *d_out_off, uint8_t *d_bytes, int64_t capacity,
                               int64_t *total_bytes, void *stream);

/* ---- small public helpers of the class, also run on the device ------------------------------- */
/* Tokenize.bpe(token) (tokenize.py:62-101): piece_cp[i] = code points in piece i of the word. */
int genztok_bpe_word(genztok_t *h, const uint8_t *word, int64_t word_len, int32_t *piece_cp, int64_t cap,
                     int64_t *n_pieces);
/* get_sequence_id (tokenize.py:163-182), optionally followed by get_token_type (:154-161), on one
 * id list.  out needs n entries (int8, GENZTOK_NONE = None).  *status = 1 when get_token_type raises. */
int genztok_sequence_id(genztok_t *h, const int32_t *ids, int64_t n, int apply_token_type, int8_t *out,
                        int64_t *out_len, int *status);
/* get_atttention_mask (tokenize.py:148-152) */
int genztok_attention_mask(genztok_t *h, const int32_t *ids, int64_t n, uint8_t *out);

/* ---- text normalisers of genz_tokenize/preprocess.py, the optional step before Tokenize (SURVEY.md 8 f3) ------ */
#define GENZTOK_PREP_REMOVE_HTML 0        /* remove_html        preprocess.py:5-9   */
#define GENZTOK_PREP_CONVERT_UNICODE 1    /* convert_unicode    preprocess.py:30-36 */
#define GENZTOK_PREP_REMOVE_PUNCTUATIONS 2 /* remove_punctuations preprocess.py:39-44 */
#define GENZTOK_PREP_REMOVE_EMOJI 3       /* remove_emoji       preprocess.py:47-72 */
#define GENZTOK_PREP_REMOVE_URL 4         /* remove_URL         preprocess.py:75-80 */
/* One normaliser over a batch of documents (packed UTF-8 + offsets in, the same out). */
int genztok_preprocess(genztok_t *h, int op, const uint8_t *text, const int64_t *text_off, int64_t n, genztok_text_t *out);
/* Device form: text in, text out, both on the device, on `stream` -- the result can go straight into genztok_encode_device.
 * Step 1 (d_out == NULL): fills d_out_off[n+1], returns the total in *total_bytes (synchronises).  Step 2: writes the text
 * (the caller allocates total + 32 bytes, 16-byte aligned, so that the encoder's 16-byte loads stay inside). */
int genztok_preprocess_device(genztok_t *h, int dev, int op, const uint8_t *d_text, const int64_t *d_text_off, int64_t n,
                              int64_t *d_out_off, uint8_t *d_out, int64_t *total_bytes, void *stream);

/* ---- utilities -------------------------------------------------------------------------------- */
void *genztok_host_alloc(size_t bytes); /* pinned host memory for inputs */
void genztok_host_free(void *p);
int genztok_device_count(const genztok_t *h);
int genztok_cache_reset(genztok_t *h);                    /* drop the device word cache */
int64_t genztok_launch_count(const genztok_t *h);         /* kernels launched by this handle so far */
/* Per-kernel CUDA-event timing (off by default).  The report is a JSON object
 * {"kernel": {"launches": L, "ms": T}, ...}; returns the length needed. */
int genztok_set_profiling(genztok_t *h, int on);
int64_t genztok_profile_report(genztok_t *h, char *buf, int64_t cap, int reset);
/* Engine knobs (see DESIGN.md).  Sizing: "max_chunk_bytes" (before the first encode; the largest chunk a call may hand over: the
 * word cache is sized for the worst case of the largest chunk met so far, up to this), "fixed_cache" (1: size it for
 * max_chunk_bytes at once), "chunk_rows".  Pipeline selection and test knobs, all defaulting to the fastest correct setting: "no_flat" (1: fused row kernel
 * even where the byte-parallel pipeline applies), "no_tma" (store instructions instead of the TMA unit), "no_fixed_decode" (fixed-width rows through the any-rows decode kernels),
 * "no_token_decode" (ragged rows decoded by a warp per row instead of a thread per id), "tma_columns" (staged
 * columns per row, multiple of 16, 0 = from the text size), "no_side_pads", "flat_rows" (rows per tile of k_flat_rows, 1..32),
 * "rows_minb" / "words_minb" / "rows_grid" (occupancy of the pipeline's kernels), "group" (documents per tile of the fused
 * kernel, 0 = auto), "wide_rows", "grid_mult", "no_stage32" (1: never narrow the staged columns to 32 by the previous call's row
 * lengths), "no_discovery" (1: no byte-parallel word pass in front of the fused row kernel on an empty cache), "decode_write"
 * (fixed-width decode, write pass: 0 = by the rows' average lead, 1 = warp per row, 2 / 3 = lane per junction with 256 / 512 bytes),
 * "decode_wide_max" (average lead up to which the 512-byte junctions are taken), "copy_round", "copy_blocks", "no_copy_kernel"
 * (host path: how the result columns travel back).  Unknown names are an error. */
int genztok_set_option(genztok_t *h, const char *name, int64_t value);

/* Error counter of the asynchronous device path (genztok_encode_device / genztok_decode_device do not synchronise, so they
 * cannot report what the kernels find: offsets outside the stated text, exhausted work lists).  Synchronises `stream`;
 * *n_errors = inconsistencies counted since the handle was created; returns GENZTOK_E_CUDA when it is not zero. */
int genztok_check_errors(genztok_t *h, int dev, void *stream, int64_t *n_errors);

/* ---- the step behind the tokenizer (SURVEY.md 8 f4) ----------------------------------------------------------------
 * DataCollection.to_tf_dataset (genz_tokenize/models/bert/dataset.py:28-55) shuffles the whole collection and cuts it into
 * batches of ({field: rows}, y).  For fields that stay on the device one launch gathers a batch of every field:
 * d_out[f][i, :] = d_fields[f][d_index[i], :] for f < n_fields (<= GENZTOK_MAX_FIELDS), row_bytes[f] bytes per row of field f,
 * n_rows rows per field, d_index[n_index] on the device (a number outside [0, n_rows) gives a row of zero bytes).  Does not
 * synchronise. */
#define GENZTOK_MAX_FIELDS 8
int genztok_gather_rows(genztok_t *h, int dev, int n_fields, const void *const *d_fields, const int64_t *row_bytes,
                        int64_t n_rows, const int64_t *d_index, int64_t n_index, void *const *d_out, void *stream);

/* ---- measurement plumbing (not part of the reference's surface; used by bench.py and the tests) ------------------- */
/* The synthetic workload of SURVEY.md 8 d2 produced on the device: the counter-based generator that
 * genz_tokenize_b200/workload.py::generate_hashed defines (same bytes).  genztok_synth_init uploads the word list
 * (packed words, start / length per word, 32-bit CDF of their counts) and the glue pieces of the noise words.
 * genztok_synth_device, step 1 (d_bytes == NULL): byte offsets of documents [doc0, doc0 + n) of `side` into d_off[n+1],
 * total in *total_bytes (synchronises); step 2: the bytes. */
int genztok_synth_init(genztok_t *h, int dev, const uint8_t *wblob, int64_t wblob_len, const uint32_t *wstart,
                       const uint32_t *wlen, const uint32_t *cdf32, int64_t nw, const uint8_t *eblob, int64_t eblob_len,
                       const uint32_t *estart, const uint32_t *elen, int64_t ne);
int genztok_synth_device(genztok_t *h, int dev, uint64_t seed, int64_t doc0, int64_t n, int side, int lo, int hi,
                         uint32_t noise_thr, int64_t *d_off, uint8_t *d_bytes, int64_t *total_bytes, void *stream);
/* Order-independent digest of fixed-layout planes on the device: *d_acc += sum over rows r and 32-bit words i of
 * mix64((mix64((row0 + r) * GOLD) + (plane << 32 | i) * GOLD) ^ word), planes 0 = input_ids, 1 = attention_mask,
 * 2 = token_type_ids (NULL: skipped).  Equal for any sharding / chunking of the same batch (SURVEY.md 8 d7). */
int genztok_digest_device(genztok_t *h, int dev, const int32_t *d_ids, const uint8_t *d_mask, const int8_t *d_tt,
                          int64_t n, int32_t width, int64_t row0, uint64_t *d_acc, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GENZTOK_H */
