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
/* Pair truncation strategies (HF's truncation="longest_first" / "only_first" / "only_second"), for genztok_encode and
 * genztok_encode_device; at most one.  Without them, truncation cuts the concatenation [bos] A [eos eos] B [eos] to max_len and
 * forces a final </s> (tokenize.py:141-146), which can drop all of B.  With la, lb the untruncated token counts of the two texts
 * (len(encode(x)) - 2) and C = max_len - 4:
 *  - la + lb <= C: every strategy gives the row of the reference cut, on every plane.
 *  - LONGEST_FIRST, the rule of the Rust `tokenizers` library (HF's fast tokenizers, truncate_encodings / LongestFirst): the
 *    shorter text (the first when la == lb) stays whole when it has at most floor(C/2) tokens and the longer keeps C - shorter;
 *    otherwise the shorter keeps floor(C/2) and the longer ceil(C/2).  At C = 9: (3, 20) -> (3, 6), (20, 3) -> (6, 3),
 *    (10, 10) -> (4, 5), (20, 10) -> (5, 4).  (HF's Python "slow" tokenizers break the tie the other way: (10, 10) -> (5, 4).)
 *  - ONLY_SECOND: A stays whole and B keeps C - la tokens, when la < C.  ONLY_FIRST: B stays whole and A keeps C - lb, when
 *    lb < C.  Otherwise (HF raises SequenceTooShort) the row's row_status is 2 and its planes hold the reference cut's row.
 * The kept tokens form [bos] + A[:la'] + [eos, eos] + B[:lb'] + [eos] (at most max_len entries), which then goes through the
 * reference's padding, attention mask, get_sequence_id and get_token_type unchanged: a row of exactly max_len entries gets the
 * </s>-id last token type, and row_status 1 happens only where those rules raise on that list (a literal <s> / </s> word in a
 * text).  With GENZTOK_WANT_OFFSETS (host form) a kept token has its untruncated offsets, everything else (0, 0).  Requires
 * max_len >= 4 and, for genztok_encode, padding, truncation and no GENZTOK_WANT_SPANS; otherwise GENZTOK_E_INVALID, reported
 * before the device is looked at.  A batch without second texts ignores the strategy. */
#define GENZTOK_LONGEST_FIRST 16u
#define GENZTOK_ONLY_FIRST 32u
#define GENZTOK_ONLY_SECOND 64u

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
    uint8_t *row_status;     /* [n] or NULL; 1 = the reference raises ValueError (tokenize.py:157-159); 2 = the pair truncation
                              * strategy of the call cannot apply (HF's SequenceTooShort; takes precedence over 1) */
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
 * genztok_encode_windows_device: window 0 of each document (rows d_win_off[:-1]) is its genztok_encode row.
 * A pair truncation strategy (GENZTOK_LONGEST_FIRST / _ONLY_FIRST / _ONLY_SECOND, with pairs) needs input_ids, attention_mask and
 * row_len, and synchronises: the token streams of the two texts are sized by reading their length back from the device, once per
 * text, before the rows are written. */
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

/* ---- extractive question answering over the windows' planes (the targets and outputs of the reference's QA models) ---------
 * Both read the offset_mapping plane d_offsets [n_windows][max_len][2] of genztok_encode_windows(_device) (or of a fixed-layout
 * genztok_encode, one window per document: d_win_off = 0, 1, ..., n) and d_win_off [n_docs + 1]; windows win_off[d] .. win_off[d+1]-1
 * belong to document d, whose answer lives in the windowed text (the second text of pairs).
 * Context columns of a window, from the offsets alone (token types move with a question that holds a literal </s>): singles,
 * every column with end > 0; pairs, with z the first column >= 1 that is (0, 0), the columns after z with end > 0.  They form
 * one range of columns, possibly empty (a pair whose question fills the row has none).
 * Labels: with the answer [a0, a1) in bytes of the document, cols = the context columns with start < a1 and end > a0; the
 * window's label is (cols[0], cols[-1]) when cols is not empty, start(cols[0]) <= a0 and end(cols[-1]) >= a1, else (0, 0) (the <s>
 * column).  a1 <= a0 ("no answer") and spans past the document's end give (0, 0) in every window; an answer inside the stride
 * overlap is labelled in every window that wholly holds it.  GENZTOK_QA_CHARS: d_answers are indices into the Python str; index
 * k becomes the byte of the code point with index k (a code point is a byte that is not 10xxxxxx: Python's count for
 * 'surrogatepass' UTF-8), the character count becomes the byte length, a larger index the byte length plus the excess (past
 * the end), a negative one stays as it is.  The text (d_text 16-byte aligned and readable to a multiple of 16 bytes,
 * d_text_off[n_docs + 1]) is what was windowed.  One launch per call (two with characters).
 * Best spans: candidates (i, s, e) with i a window of d, s <= e context columns of i and e - s + 1 <= max_answer_len; score
 * start_logits[i][s] + end_logits[i][e] (one float add).  The best is the largest score, ties to the smallest i, then s, then e;
 * a NaN score is never taken.  This is the exact maximum over every valid pair (HF's top-20 x top-20 pre-filter can only find a
 * lower or equal one).  Per document: d_score, d_window (global window index), d_columns (s, e), d_span = (start of s, end of e),
 * the answer's byte range in the document, and d_null_score = the fminf over its windows of start_logits[i][0] + end_logits[i][0]
 * (SQuAD v2's "no answer" score).  A document without a candidate gets window -1, score -inf, columns = span = (0, 0).  A warp
 * stages its window's two logit rows in shared memory: max_len above the device's per-block limit / 16 bytes is GENZTOK_E_LIMIT.
 * Two launches per call.
 * Both are asynchronous on `stream` of device slot `dev` and bit-identical from run to run.  Offsets that break the layout and a
 * win_off that does not fit n_windows are counted by genztok_check_errors (such windows get (0, 0) and no candidate). */
#define GENZTOK_QA_BYTES 0
#define GENZTOK_QA_CHARS 1
int genztok_qa_labels_device(genztok_t *h, int dev, const int32_t *d_offsets, int64_t n_windows, int32_t max_len, int has_pair,
                             const int64_t *d_win_off, int64_t n_docs, const int64_t *d_answers /* [n_docs][2] */, int unit,
                             const uint8_t *d_text, const int64_t *d_text_off, int64_t text_bytes /* GENZTOK_QA_CHARS only */,
                             int64_t *d_start, int64_t *d_end /* [n_windows] */, void *stream);
int genztok_qa_best_spans_device(genztok_t *h, int dev, const float *d_start_logits, const float *d_end_logits /* [n_windows][max_len] */,
                                 const int32_t *d_offsets, int64_t n_windows, int32_t max_len, int has_pair, const int64_t *d_win_off,
                                 int64_t n_docs, int32_t max_answer_len, float *d_score, float *d_null_score, int64_t *d_window,
                                 int32_t *d_columns /* [n_docs][2] */, int32_t *d_span /* [n_docs][2] */, void *stream);

/* ---- masked-language-model inputs and labels (the pre-training recipe of the reference's RoBERTa / DistilBERT models) ------
 * Reads a fixed-layout id plane d_ids [n][width] (any encode, window or gathered batch) and writes d_masked_ids [n][width] (int32)
 * and d_labels [n][width] (int64): at a selected column the replaced id and the original id, everywhere else the input id and
 * -100 (HF's DataCollatorForLanguageModeling conventions).  d_ids is not modified; d_masked_ids must not be d_ids.
 *  - Eligible column: 0 <= id < n_ids (the size of the handle's id table) and id is none of the five special ids.  Framing, pads,
 *    an existing mask, unk and ids the vocab does not know are never selected, so every label is -100 or a valid class index.
 *  - Continuation id: an id in the decoder whose string ends in the two bytes "@@" (the pieces decode glues to the next piece);
 *    no other id continues, including ids absent from the decoder and ids outside [0, n_ids).
 *  - Group of column j: j itself; with whole_word, the largest g <= j with g == 0 or ids[r][g - 1] not a continuation id.  A group
 *    can hold ineligible columns (a word cut by truncation runs into the forced </s>).  Selection is decided per group and
 *    applies to the group's eligible columns.
 *  - Hashes, mod 2^64, with mix64 the splitmix64 finaliser, GOLD = 0x9E3779B97F4A7C15, K = 0x6D6C6D5F6D61736B and key_r =
 *    d_row_keys[r] (NULL: r):  R_r = mix64(mix64(seed ^ K) + key_r * GOLD).  Column j of row r is selected when it is eligible
 *    and (mix64(R_r + (2 g(j) + 1) * GOLD) >> 32) < T_sel.  A selected column draws v = mix64(R_r + (2 j + 2) * GOLD), u = v >> 32:
 *    u < T_mask gives the mask id, else u < T_mask_rand gives repl[((v & 0xFFFFFFFF) * M) >> 32], else the id is kept.  With
 *    p = mlm_probability, a = mask_replace_prob, b = random_replace_prob (HF's names; 0.15, 0.8, 0.1 are HF's defaults):
 *    T_sel = floor(p * 2^32), T_mask = floor(a * 2^32), T_mask_rand = floor((a + b) * 2^32), computed in double, so p = 1 selects
 *    every eligible column and p = 0 none.  repl is the ascending list of the M ids that are in the decoder and not special.
 * Differences from HF: selection is a Bernoulli draw per group (HF's whole-word collator draws an exact count per row); random
 * replacements exclude the special ids (HF's randint(len(tokenizer)) includes them); the result is a pure function of (seed,
 * key, row contents), independent of batch composition, sharding and any other RNG -- dynamic masking takes a new seed per
 * epoch.  Windows that overlap draw independent decisions for the tokens they share (their rows and keys differ).
 * Checks: the probabilities finite and in [0, 1], a + b <= 1, n >= 0, width >= 1, non-NULL pointers when n > 0, d_masked_ids
 * != d_ids, and b > 0 only with M > 0 (GENZTOK_E_INVALID), all before the device slot.  Asynchronous on `stream`, one launch
 * per call (none when n == 0), bit-identical from run to run.  The first call on a device uploads the continuation bitset
 * (n_ids / 8 bytes) and repl (4 M bytes). */
int genztok_mlm_mask_device(genztok_t *h, int dev, const int32_t *d_ids, int64_t n, int32_t width,
                            const int64_t *d_row_keys /* NULL: row index */, uint64_t seed,
                            double mlm_probability, double mask_replace_prob, double random_replace_prob,
                            int whole_word, int32_t *d_masked_ids, int64_t *d_labels, void *stream);

/* ---- BPE-dropout (Provilkov et al., 2020): a different segmentation of the same text on every epoch --------------------
 * Fixed-layout rows (padding, the reference cut, max_len >= 4) as genztok_encode gives them, except that every merge may be skipped.
 * Words are split as always: the \S+\n? matches of tokenize.py:106 (the 29 whitespace code points of Python's \s), each starting
 * from bpe()'s initial symbols (its code points, "</w>" on the last).  The merge loop is subword-nmt's encode() with dropout:
 *  1. in round t (from 0), the pair at position i (from 0) of the current symbol sequence is dropped when its draw says so;
 *  2. if no pair that is in bpe_ranks survives, the word is final (a round that drops every candidate ends the word; it is not
 *     retried);
 *  3. else the surviving pair with the lowest rank is merged at its surviving occurrences, left to right, an occurrence that overlaps
 *     one merged before it in the round being skipped (x x x -> xx x); dropped occurrences of that pair stay unmerged;
 *  4. until one symbol is left.  Pieces map to ids as always (S + "@@" / S[:-4], unk when the vocab lacks the piece).
 * With p = 0 this is bpe(): the rows are bit-identical to genztok_encode's on every plane.  With p = 1 every word is its code points,
 * which are unk unless the vocab holds each code point with and without "@@".  HF tokenizers' BPE(dropout=p) puts dropped merges
 * back after the next successful merge and so gives other segmentations.
 * Draws, mod 2^64, with mix64 the splitmix64 finaliser, GOLD = 0x9E3779B97F4A7C15 and K = 0x6270655F64726F70 ("bpe_drop"):
 *    s0 = mix64(seed ^ K);  R = mix64(s0 + key * GOLD);  W_j = mix64(R + (2 j + side + 1) * GOLD);
 *    pair (t, i) of word j is dropped  <=>  (mix64(W_j + (t << 32 | i)) >> 32) < floor(p * 2^32)  (computed in double; p = 1 drops all)
 * with key = row_keys[r] (NULL: the row's index in the whole call), j the index of the word among its text's \S+\n? matches and
 * side 0 for the text, 1 for the second text.  The rows are a pure function of (seed, key, text): they do not depend on chunking,
 * sharding over the handle's devices, batch order (with keys that follow the documents) or the word cache, which is neither read
 * nor written.  A text's words are merged only until it has max_len ids: the reference cut shows no more of it.
 * Checks, before the device slot (GENZTOK_E_INVALID): n >= 0, p in [0, 1] (not NaN), max_len >= 4, and flags among
 * GENZTOK_WANT_TOKEN_TYPE | GENZTOK_WANT_SEQUENCE_ID (offsets, spans and the pair truncation strategies are not available).
 * genztok_encode_dropout: host buffers, results as genztok_encode's fixed layout (free with genztok_free_encoded), chunked and
 * sharded as genztok_encode.  genztok_encode_dropout_device: everything on device `dev`, asynchronous on `stream` with no host read
 * (planes: input_ids, attention_mask and row_len required; pairs also write seq_len / row_status when given); its work buffers grow
 * (cudaMalloc / cudaFree) only on a call larger than every earlier one on the device.  Both use n * (max_len + 2) * 4 bytes per side
 * of device memory for the capped token streams and 8 bytes per text byte of scratch for long words (released by genztok_destroy).
 * A document whose offsets do not lie inside its side's bytes is counted by genztok_check_errors (the host form fails with
 * GENZTOK_E_CUDA) and gets no ids.
 * genztok_bpe_word_dropout: genztok_bpe_word under dropout, the segmentation of word 0, side 0 of a row with key `key`. */
int genztok_encode_dropout(genztok_t *h, const uint8_t *text, const int64_t *text_off, const uint8_t *pair, const int64_t *pair_off, int64_t n,
                           int32_t max_len, uint32_t flags, double p, uint64_t seed, const int64_t *row_keys /* [n] or NULL */,
                           genztok_encoded_t *out);
int genztok_encode_dropout_device(genztok_t *h, int dev, const uint8_t *d_text, const int64_t *d_text_off, int64_t text_bytes,
                                  const uint8_t *d_pair, const int64_t *d_pair_off, int64_t pair_bytes, int64_t n, int32_t max_len,
                                  uint32_t flags, double p, uint64_t seed, const int64_t *d_row_keys /* [n] or NULL */,
                                  const genztok_dev_planes_t *planes, void *stream);
int genztok_bpe_word_dropout(genztok_t *h, const uint8_t *word, int64_t word_len, double p, uint64_t seed, int64_t key,
                             int32_t *piece_cp, int64_t cap, int64_t *n_pieces);

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
