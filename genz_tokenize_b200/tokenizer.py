"""`Tokenize`: the reference's public class (genz_tokenize/tokenize.py:6-267) as a thin ctypes
wrapper over libgenztok.so.  Same constructor, `fromFile`, `__call__`, `encode`, `decode`, `bpe`,
`vocab_size`, helper methods and attributes; every tokenisation step runs in CUDA kernels on a
B200 -- there is no CPU path, and a handle without a device raises.

Extensions over the reference (which is one string per call): `encode_batch` / `decode_batch`
(numpy in, numpy out through pinned host buffers), `encode_device` / `decode_device`
(torch CUDA tensors in and out, DLPack-exportable, nothing crosses PCIe) and `encode_windows` /
`encode_windows_device` (long documents as overlapping max_len windows, every token kept).  Every encode
form but encode_device can also return `offset_mapping` (HF's return_offsets_mapping): each token's
(start, end) byte range in its own document's UTF-8 text, (0, 0) for tokens that are not from the text.
`truncation=` also takes HF's pair strategies "longest_first", "only_first" and "only_second" (fixed layout).
`qa_labels` / `qa_best_spans` turn those planes into extractive-QA training labels and read a QA model's
start / end logits back into answer spans, on the GPU.  `mlm_mask` turns any fixed-layout id plane into masked-language-model
inputs and labels (token or whole-word masking), on the GPU.  `bpe_dropout=p` on encode_batch / encode_device (and `dropout=p` on
`bpe`) skips every merge with probability p (BPE-dropout), a different segmentation per seed, on the GPU.
"""
import ctypes as C
import operator
import os

import numpy as np

from . import _lib as L
from .data import bundled_paths


class GenztokError(RuntimeError):
    pass


# truncation= names of the pair truncation strategies (include/genztok.h states the rule)
_STRATEGIES = {"longest_first": L.LONGEST_FIRST, "only_first": L.ONLY_FIRST, "only_second": L.ONLY_SECOND}


def _strategy_flag(truncation, max_len, padding=True, return_offset=False):
    """The flag of a strategy name, after the checks of the fixed layout it needs; 0 for anything that is not a str."""
    if not isinstance(truncation, str):
        return 0
    if truncation not in _STRATEGIES:
        raise ValueError("truncation must be True, False or one of %s (got %r)" % (", ".join(map(repr, _STRATEGIES)), truncation))
    if max_len is None or max_len < 4:
        raise ValueError("truncation=%r needs max_len >= 4 (got %r)" % (truncation, max_len))
    if not padding:
        raise ValueError("truncation=%r needs padding=True (the fixed layout)" % truncation)
    if return_offset:
        raise ValueError("truncation=%r is not available with return_offset=True" % truncation)
    return _STRATEGIES[truncation]


def _dropout_args(bpe_dropout, seed, max_len, padding=True, truncation=True, return_offset=False, return_offsets_mapping=False):
    """(p, seed as uint64) of a BPE-dropout encode, after the checks of the fixed layout it needs."""
    p = float(bpe_dropout)
    if not 0.0 <= p <= 1.0:
        raise ValueError("bpe_dropout must be in [0, 1] (got %r)" % bpe_dropout)
    if max_len is None or max_len < 4:
        raise ValueError("bpe_dropout needs max_len >= 4 (got %r)" % (max_len,))
    if not padding:
        raise ValueError("bpe_dropout needs padding=True (the fixed layout)")
    if truncation is not True:
        raise ValueError("bpe_dropout needs truncation=True (the reference cut; got %r)" % (truncation,))
    if return_offset or return_offsets_mapping:
        raise ValueError("bpe_dropout is not available with return_offset / return_offsets_mapping")
    return p, operator.index(seed) & (2 ** 64 - 1)


def pack_strings(strs):
    """list[str] -> (uint8 bytes, int64 offsets[n+1]) in the ABI's UTF-8 ('surrogatepass') form."""
    enc = []
    for s in strs:
        if not isinstance(s, str):
            raise TypeError("expected string or bytes-like object, got %r" % type(s).__name__)   # re.findall, tokenize.py:106
        enc.append(s.encode("utf-8", "surrogatepass"))
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    if enc:
        np.cumsum(np.fromiter((len(e) for e in enc), dtype=np.int64, count=len(enc)), out=off[1:])
    blob = b"".join(enc)
    return np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(0, dtype=np.uint8), off


def _view(ptr, count, ctype, dtype, owner):
    """Zero-copy numpy view of library-owned memory; `owner` is kept alive by the array's base."""
    if count == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    buf = (ctype * count).from_address(C.addressof(ptr.contents))
    buf._owner = owner
    return np.frombuffer(buf, dtype=dtype)


class _EncodedOwner:
    def __init__(self, tok, enc, free="genztok_free_encoded"):
        self.tok, self.enc, self.free = tok, enc, free

    def __del__(self):
        try:
            if self.tok._h:
                getattr(self.tok._lib, self.free)(self.tok._h, C.byref(self.enc))
        except Exception:
            pass


class BatchEncoding(dict):
    """dict of numpy arrays.  Fixed layout: [n, max_len] arrays.  Ragged layout: flat arrays plus
    'row_off' (int64[n+1]).  `row(i)` gives the reference's per-call dict for row i."""

    def row(self, i):
        return self._tok._row_to_dict(self, i)


class Tokenize(object):
    def __init__(self, pad_token='<pad>', bos_token='<s>', eos_token='</s>', mask_token='<mask>', unk_token='<unk>',
                 *, devices=None):
        super().__init__()
        # tokenize.py:15-23: fromFile pre-sets the two paths, otherwise the bundled files are used
        if not hasattr(self, 'vocab_file') or not hasattr(self, 'bpe_file'):
            v, b = bundled_paths()
            if not hasattr(self, 'vocab_file'):
                self.vocab_file = v
            if not hasattr(self, 'bpe_file'):
                self.bpe_file = b
        self.pad_token = pad_token
        self.bos_token = bos_token
        self.eos_token = eos_token
        self.mask_token = mask_token
        self.unk_token = unk_token
        self._devices = devices
        self._extra_vocab = []
        if getattr(self, "_h_dec", None):
            self._close_decoder()
        self._h = self._h_dec = None
        self._open()

    # ---- handle management ---------------------------------------------------------------------
    def _open(self):
        self._close()
        self._lib = L.load()
        devices = self._devices
        if devices is None:
            devices = [int(os.environ.get("GENZTOK_DEVICE", os.environ.get("LOCAL_RANK", "0")))]
        for t in (self.pad_token, self.bos_token, self.eos_token, self.mask_token, self.unk_token):
            if not isinstance(t, str):
                raise TypeError("special tokens must be str")
        sp = (C.c_char_p * 5)(*[t.encode("utf-8", "surrogatepass") for t in
                                (self.pad_token, self.bos_token, self.eos_token, self.mask_token, self.unk_token)])
        dev = (C.c_int * max(len(devices), 1))(*devices)
        self._device_ids = list(devices)
        h = C.c_void_p()
        vocab = self.vocab_file
        if self._extra_vocab:
            vocab = self._merged_vocab()
        rc = self._lib.genztok_create(os.fsencode(vocab), os.fsencode(self.bpe_file), sp, dev, len(devices), C.byref(h))
        if self._extra_vocab:                                   # the merged copy was only for the loader
            try:
                os.unlink(vocab)
            except OSError:
                pass
        if rc:
            msg = (self._lib.genztok_last_error(None) or b"").decode("utf-8", "replace")
            if rc == L.E_IO:
                raise FileNotFoundError(msg)
            if rc == L.E_UTF8:
                raise UnicodeDecodeError("utf-8", b"", 0, 1, msg)
            raise GenztokError("genztok_create failed (%d): %s -- the tokenizer needs a CUDA device; there is no CPU path" % (rc, msg))
        self._h = h
        self._ids = None
        self._encoder = self._decoder = self._bpe_ranks = None
        if getattr(self, "_h_dec", None):
            self._decoder = self._decoder_frozen
        for k, v in getattr(self, "_options", {}).items():
            self._set_option(k, v)

    def _close(self):
        if getattr(self, "_h", None):
            self._lib.genztok_destroy(self._h)
        self._h = None

    def _close_decoder(self):
        if getattr(self, "_h_dec", None):
            self._lib.genztok_destroy(self._h_dec)
        self._h_dec = None

    @property
    def _hd(self):
        """The handle whose tables `decode` reads: the one built by __init__ (tokenize.py:40 builds `decoder` there and nothing
        refreshes it: add_vocab_file after construction leaves it stale), else the current one."""
        return getattr(self, "_h_dec", None) or self._h

    def __del__(self):
        try:
            self._close()
            self._close_decoder()
        except Exception:
            pass

    def _err(self, rc, what):
        msg = (self._lib.genztok_last_error(self._h) or b"").decode("utf-8", "replace")
        raise GenztokError("%s failed (%d): %s" % (what, rc, msg))

    def _set_option(self, name, value):
        rc = self._lib.genztok_set_option(self._h, name.encode(), int(value))
        if rc:
            self._err(rc, "genztok_set_option(%s)" % name)

    def set_option(self, name, value):
        """Engine knob (max_chunk_bytes, chunk_rows, group); remembered across re-initialisation."""
        self._set_option(name, value)
        self.__dict__.setdefault("_options", {})[name] = value

    # ---- tables as the reference's attributes ------------------------------------------------------
    def _special_ids(self):
        if self._ids is None:
            out = (C.c_int32 * 5)()
            self._lib.genztok_special_ids(self._h, out)
            self._ids = list(out)
        return self._ids

    @property
    def encoder(self):
        if self._encoder is None:
            d = {}
            key, klen, vid = C.POINTER(C.c_uint8)(), C.c_int64(), C.c_int32()
            for i in range(self._lib.genztok_encoder_count(self._h)):
                self._lib.genztok_encoder_entry(self._h, i, C.byref(key), C.byref(klen), C.byref(vid))
                d[C.string_at(key, klen.value).decode("utf-8", "surrogatepass")] = vid.value
            self._encoder = d
        return self._encoder

    @property
    def decoder(self):
        if self._decoder is None:
            self._decoder = {v: k for k, v in self.encoder.items()}      # tokenize.py:40
        return self._decoder

    @property
    def bpe_ranks(self):
        if self._bpe_ranks is None:
            d = {}
            line, ln = C.POINTER(C.c_uint8)(), C.c_int64()
            for i in range(self._lib.genztok_merge_count(self._h)):
                self._lib.genztok_merge_line(self._h, i, C.byref(line), C.byref(ln))
                d[tuple(C.string_at(line, ln.value).decode("utf-8", "surrogatepass").split())] = i   # tokenize.py:56-57
            self._bpe_ranks = d
        return self._bpe_ranks

    def vocab_size(self):
        return int(self._lib.genztok_vocab_size(self._h))                # tokenize.py:59-60

    def _merged_vocab(self):
        import tempfile
        parts = []
        for p in [self.vocab_file] + self._extra_vocab:
            with open(p, "rb") as f:
                b = f.read()
            if b and not b.endswith((b"\n", b"\r")):
                b += b"\n"
            parts.append(b)
        fd, path = tempfile.mkstemp(prefix="genztok_vocab_", suffix=".txt")
        with os.fdopen(fd, "wb") as f:
            f.write(b"".join(parts))
        self._tmp_vocab = path
        return path

    def add_vocab_file(self, vocab_file):
        """tokenize.py:44-51: append another vocab file's words to `encoder` (the device tables are rebuilt).  `decoder` is NOT
        refreshed by the reference (it is built once, tokenize.py:40): ids added here decode to the unk token, and a word that
        moved keeps decoding from its old id.  The handle of the tables as __init__ built them is kept for decoding."""
        with open(vocab_file, 'r', encoding='utf-8'):
            pass
        self._extra_vocab.append(vocab_file)
        if getattr(self, "_h_dec", None) is None:
            self._decoder_frozen = self.decoder                   # the dict as of construction
            self._h_dec, self._h = self._h, None                  # (kept alive: _open() destroys only self._h)
        self._open()
        self._decoder = self._decoder_frozen

    def add_bpe_file(self, bpe_file):
        """tokenize.py:53-57: replace the merge table (the device tables are rebuilt)."""
        with open(bpe_file, 'r', encoding='utf-8'):
            pass
        self.bpe_file = bpe_file
        self._open()

    # ---- single-call surface ---------------------------------------------------------------------------
    def bpe(self, token, dropout=None, seed=0, key=0):
        """tokenize.py:62-101 -- the merge loop runs on the device; pieces are cut from `token` by code point.  dropout=p: the
        BPE-dropout segmentation (include/genztok.h) of `token` as the first word of a row with row key `key`, encoded with `seed`."""
        if not isinstance(token, str):
            token = "".join(token)
        if len(token) == 0:
            raise IndexError("tuple index out of range")                 # word[-1] on an empty tuple, :64
        w = token.encode("utf-8", "surrogatepass")
        cap = len(token) + 1
        pieces = (C.c_int32 * cap)()
        n = C.c_int64()
        if dropout is None:
            rc = self._lib.genztok_bpe_word(self._h, w, len(w), pieces, cap, C.byref(n))
        else:
            p = float(dropout)
            if not 0.0 <= p <= 1.0:
                raise ValueError("dropout must be in [0, 1] (got %r)" % dropout)
            rc = self._lib.genztok_bpe_word_dropout(self._h, w, len(w), p, operator.index(seed) & (2 ** 64 - 1), operator.index(key), pieces, cap, C.byref(n))
        if rc:
            self._err(rc, "genztok_bpe_word")
        out, pos = [], 0
        for i in range(n.value):
            out.append(token[pos:pos + pieces[i]])
            pos += pieces[i]
        return "@@ ".join(out)

    def encode(self, sentence, return_offset):
        """tokenize.py:126-135"""
        if not isinstance(sentence, str):
            raise TypeError("expected string or bytes-like object, got %r" % type(sentence).__name__)
        r = self._encode_raw([sentence], None, None, True, True, 0, return_offset)
        ids = r["input_ids"].tolist()
        if return_offset:
            return ids, [tuple(p) for p in r["spans"].tolist()]
        return ids

    def decode(self, token):
        """tokenize.py:137-139"""
        ids = self._ids_to_int32(token)
        return self.decode_batch(ids, np.array([0, len(ids)], dtype=np.int64))[0]

    def get_atttention_mask(self, token):
        """tokenize.py:148-152"""
        ids = self._ids_to_int32(token, unknown=self._non_pad_id())
        out = np.zeros(len(ids), dtype=np.uint8)
        rc = self._lib.genztok_attention_mask(self._h, ids.ctypes.data, len(ids), out.ctypes.data)
        if rc:
            self._err(rc, "genztok_attention_mask")
        return [int(v) for v in out]

    def get_sequence_id(self, token):
        """tokenize.py:163-182"""
        return self._sequence_id(token, False)

    def get_token_type(self, token):
        """tokenize.py:154-161 (mutates and returns its argument)"""
        token[0] = 0
        token[-1] = 1
        index = token.index(None)
        token[index] = 0
        index = token.index(None)
        token[index] = 1
        return token

    def _non_pad_id(self):
        pad = self._special_ids()[0]
        return 0 if pad != 0 else 1

    def _sequence_id(self, token, apply_token_type):
        ids = self._ids_to_int32(token, unknown=-7)
        out = np.zeros(max(len(ids), 1), dtype=np.int8)
        n, st = C.c_int64(), C.c_int()
        rc = self._lib.genztok_sequence_id(self._h, ids.ctypes.data, len(ids), int(apply_token_type), out.ctypes.data, C.byref(n), C.byref(st))
        if rc:
            self._err(rc, "genztok_sequence_id")
        if st.value:
            raise ValueError("None is not in list")
        return [None if v == L.NONE else int(v) for v in out[:n.value]]

    @staticmethod
    def _ids_to_int32(token, unknown=-1):
        """Python ids -> int32; anything that cannot equal an int key of `decoder` becomes `unknown`."""
        if isinstance(token, np.ndarray) and token.dtype.kind in "iu":
            a = token.astype(np.int64, copy=False).ravel()
            return np.where((a < 0) | (a > 2 ** 31 - 1), unknown, a).astype(np.int32)
        out = []
        for x in token:
            v = unknown
            try:
                i = int(x)
                if i == x and hash(i) == hash(x) and 0 <= i <= 2 ** 31 - 1:
                    v = i
            except (TypeError, ValueError, OverflowError):
                pass
            out.append(v)
        return np.asarray(out, dtype=np.int32).reshape(-1)

    def __call__(self, text, pair_text=None, max_len=None, padding=True, truncation=True, return_offset=False, return_offsets_mapping=False, **kw):
        """tokenize.py:184-259.  `text_pair=` is accepted as an alias of `pair_text`.  return_offsets_mapping: also
        'offset_mapping', a (start, end) byte range per token (see encode_batch).  truncation: as encode_batch (a pair that
        a strategy cannot truncate raises ValueError)."""
        if "text_pair" in kw:
            if pair_text is not None:
                raise TypeError("pass pair_text or text_pair, not both")
            pair_text = kw.pop("text_pair")
        if kw:
            raise TypeError("__call__() got an unexpected keyword argument %r" % next(iter(kw)))
        if not isinstance(text, str):
            raise TypeError("expected string or bytes-like object, got %r" % type(text).__name__)
        if pair_text is not None and not isinstance(pair_text, str):
            raise TypeError("expected string or bytes-like object, got %r" % type(pair_text).__name__)
        if max_len is not None:
            max_len = operator.index(max_len)
        flags = (L.WANT_TOKEN_TYPE | L.WANT_SEQUENCE_ID) if pair_text is not None else 0
        if return_offsets_mapping:
            flags |= L.WANT_OFFSETS
        r = self._encode_raw([text], None if pair_text is None else [pair_text], max_len, padding, truncation, flags, return_offset)
        return self._row_to_dict(r, 0, return_offset)

    def _row_to_dict(self, r, i, return_offset=False):
        n = r._n
        if not 0 <= i < n:
            raise IndexError(i)
        if r._width > 0:
            s, e = i * r._width, (i + 1) * r._width
        else:
            s, e = int(r._row_off[i]), int(r._row_off[i + 1])
        result = {}
        if return_offset:
            so, eo = int(r._span_off[i]), int(r._span_off[i + 1])
            result['offset'] = [tuple(p) for p in r._spans[so:eo].tolist()]
        result['input_ids'] = r._ids[s:e].tolist()
        result['attention_mask'] = r._mask[s:e].tolist()
        if r._offsets is not None:
            result['offset_mapping'] = [tuple(p) for p in r._offsets[s:e].tolist()]
        if r._has_pair:
            if r._status[i] == 2:
                raise ValueError("truncation=%r cannot truncate row %d to max_len: the text it may cut is too short (HF's "
                                 "SequenceTooShort)" % (r._strategy, i))
            if r._status[i]:
                raise ValueError("None is not in list")                   # tokenize.py:157-159
            pad, _, eos = self._special_ids()[:3]
            conv = lambda a: [None if v == L.NONE else (eos if v == L.EOS_MARK else (pad if v == L.PAD_MARK else int(v))) for v in a]
            if r._seq is None or (r._pad_mode and r._tt is None):
                raise ValueError("row(): this batch was encoded without its sequence_id / token_type_ids planes (encode_batch(..., sequence_id=False / token_type_ids=False))")
            seq = conv(r._seq[s:s + int(r._seq_len[i])])
            result['sequence_id'] = seq
            if r._pad_mode:
                result['token_type_ids'] = conv(r._tt[s:s + int(r._tt_len[i])])
            else:
                result['token_type_ids'] = seq                             # same list object, tokenize.py:254-255
        return result

    def _encode_raw(self, texts, pairs, max_len, padding, truncation, flags, return_offset=False):
        tb, to = texts if isinstance(texts, tuple) else pack_strings(texts)
        n = len(to) - 1
        if pairs is not None:
            pb, po = pairs if isinstance(pairs, tuple) else pack_strings(pairs)
            if len(po) - 1 != n:
                raise ValueError("texts and pair_texts differ in length")
            pbp, pop = pb.ctypes.data, po.ctypes.data
        else:
            pb = po = None
            pbp = pop = None
        if return_offset:
            flags |= L.WANT_SPANS
        strategy = _strategy_flag(truncation, max_len, padding, return_offset)
        enc = L.Encoded()
        ml = L.MAX_LEN_NONE if max_len is None else int(max_len)
        if max_len is not None and not -(2 ** 31) < ml < 2 ** 31:
            raise OverflowError("max_len out of range")
        tb = np.ascontiguousarray(tb, dtype=np.uint8)
        to = np.ascontiguousarray(to, dtype=np.int64)
        rc = self._lib.genztok_encode(self._h, tb.ctypes.data, to.ctypes.data, pbp, pop, n, ml, int(bool(padding)), int(bool(truncation)),
                                      flags | strategy, C.byref(enc))
        if rc:
            self._err(rc, "genztok_encode")
        r = self._wrap(enc, n, max_len is not None and bool(padding), _EncodedOwner(self, enc))
        r._strategy = truncation if strategy else None
        return r

    def _wrap(self, enc, n, pad_mode, owner):
        """BatchEncoding of numpy views over the n rows of a genztok_encoded_t."""
        r = BatchEncoding()
        r._tok, r._n, r._width, r._has_pair = self, n, int(enc.width), bool(enc.has_pair)
        r._pad_mode = pad_mode
        r._strategy = None
        tot = int(enc.total)
        r._ids = _view(enc.input_ids, tot, C.c_int32, np.int32, owner)
        r._mask = _view(enc.attention_mask, tot, C.c_uint8, np.uint8, owner)
        r._row_off = _view(enc.row_off, n + 1, C.c_int64, np.int64, owner) if enc.width == 0 else None
        r._row_len = _view(enc.row_len, n, C.c_int32, np.int32, owner)
        r._tt = _view(enc.token_type_ids, tot, C.c_int8, np.int8, owner) if enc.token_type_ids else None
        r._seq = _view(enc.sequence_id, tot, C.c_int8, np.int8, owner) if enc.sequence_id else None
        r._tt_len = _view(enc.tt_len, n, C.c_int32, np.int32, owner) if enc.tt_len else None
        r._seq_len = _view(enc.seq_len, n, C.c_int32, np.int32, owner) if enc.seq_len else None
        r._status = _view(enc.row_status, n, C.c_uint8, np.uint8, owner) if enc.row_status else None
        r._offsets = _view(enc.offsets, 2 * tot, C.c_int32, np.int32, owner).reshape(-1, 2) if enc.offsets else None
        if enc.span_off:
            r._span_off = _view(enc.span_off, n + 1, C.c_int64, np.int64, owner)
            r._spans = _view(enc.spans, 2 * int(r._span_off[-1]), C.c_int32, np.int32, owner).reshape(-1, 2)
        shape = (n, r._width) if r._width > 0 else (tot,)
        r["input_ids"] = r._ids.reshape(shape)
        r["attention_mask"] = r._mask.reshape(shape)
        r["row_len"] = r._row_len
        r["real_tokens"] = int(enc.real_tokens)
        r.d2h_bytes = int(enc.d2h_bytes)
        if r._row_off is not None:
            r["row_off"] = r._row_off
        if r._has_pair:
            if r._tt is not None:
                r["token_type_ids"] = r._tt.reshape(shape)
                r["tt_len"] = r._tt_len
            if r._seq is not None:
                r["sequence_id"] = r._seq.reshape(shape)
            r["seq_len"] = r._seq_len
            r["row_status"] = r._status
        if enc.span_off:
            r["span_off"], r["spans"] = r._span_off, r._spans
        if r._offsets is not None:
            r["offset_mapping"] = r._offsets.reshape(shape + (2,))
        return r

    # ---- batch extensions -------------------------------------------------------------------------------
    def encode_batch(self, texts, pair_texts=None, max_len=None, padding=True, truncation=True, token_type_ids=True,
                     sequence_id=True, return_offset=False, return_offsets_mapping=False, bpe_dropout=None, seed=0, row_keys=None):
        """Encode n documents (or n pairs) in one call.  `texts` / `pair_texts`: list[str] or the packed
        form (uint8 bytes, int64 offsets[n+1]).  Returns a BatchEncoding of numpy arrays over pinned memory.
        return_offsets_mapping: also 'offset_mapping', int32 [n, max_len, 2] (fixed layout) or [total, 2] (ragged): the
        [start, end) byte range of each token in the UTF-8 ('surrogatepass') bytes of its own document -- `texts[i]`, or
        `pair_texts[i]` for tokens of the second text -- and (0, 0) for <s>, </s>, pads and the </s> truncation adds.
        It changes no other output.
        truncation: True / False as the reference (True cuts the concatenation <s> A </s></s> B </s> to max_len), or for pairs
        HF's "longest_first" (the Rust tokenizers' rule), "only_first" or "only_second": each text keeps a prefix so that the
        row fits max_len.  A pair that only_first / only_second cannot truncate gets row_status 2 and the True row on every
        plane; row(i) raises ValueError for it.  The strategies need max_len >= 4, padding=True and return_offset=False;
        include/genztok.h states the rule.
        bpe_dropout: None (the default) is the reference's BPE.  A probability p (0.0 included) takes the BPE-dropout path: every
        merge is skipped with probability p, drawn from (seed, row key, word, round, position) as include/genztok.h states, with
        row i's key row_keys[i] (int64 [n]) or i.  Same seed and keys, same rows; p = 0 gives the bpe_dropout=None rows.  It needs
        the fixed layout: max_len >= 4, padding=True, truncation=True, no return_offset / return_offsets_mapping."""
        flags = L.WANT_OFFSETS if return_offsets_mapping else 0
        if pair_texts is not None:
            flags |= (L.WANT_TOKEN_TYPE if token_type_ids else 0) | (L.WANT_SEQUENCE_ID if sequence_id else 0)
        if max_len is not None:
            max_len = operator.index(max_len)
        if bpe_dropout is not None:
            p, seed = _dropout_args(bpe_dropout, seed, max_len, padding, truncation, return_offset, return_offsets_mapping)
            return self._encode_dropout(texts, pair_texts, max_len, flags, p, seed, row_keys)
        return self._encode_raw(texts, pair_texts, max_len, padding, truncation, flags, return_offset)

    def _encode_dropout(self, texts, pairs, max_len, flags, p, seed, row_keys):
        tb, to = texts if isinstance(texts, tuple) else pack_strings(texts)
        n = len(to) - 1
        pbp = pop = None
        if pairs is not None:
            pb, po = pairs if isinstance(pairs, tuple) else pack_strings(pairs)
            if len(po) - 1 != n:
                raise ValueError("texts and pair_texts differ in length")
            pb, po = np.ascontiguousarray(pb, dtype=np.uint8), np.ascontiguousarray(po, dtype=np.int64)
            pbp, pop = pb.ctypes.data, po.ctypes.data
        keys = None
        if row_keys is not None:
            keys = np.ascontiguousarray(np.asarray(row_keys, dtype=np.int64))
            if keys.shape != (n,):
                raise ValueError("row_keys must have shape (%d,) (got %s)" % (n, keys.shape))
        if max_len >= 2 ** 31:
            raise OverflowError("max_len out of range")
        tb, to = np.ascontiguousarray(tb, dtype=np.uint8), np.ascontiguousarray(to, dtype=np.int64)
        enc = L.Encoded()
        rc = self._lib.genztok_encode_dropout(self._h, tb.ctypes.data, to.ctypes.data, pbp, pop, n, int(max_len), flags, p, seed,
                                              keys.ctypes.data if keys is not None else None, C.byref(enc))
        if rc:
            self._err(rc, "genztok_encode_dropout")
        return self._wrap(enc, n, True, _EncodedOwner(self, enc))

    @staticmethod
    def _window_args(max_len, stride):
        max_len, stride = operator.index(max_len), operator.index(stride)
        if max_len < 3:
            raise ValueError("encode_windows needs max_len >= 3 (got %d)" % max_len)
        if not 0 <= stride < max_len - 2:
            raise ValueError("encode_windows needs 0 <= stride < max_len - 2 (got stride=%d, max_len=%d)" % (stride, max_len))
        if max_len >= 2 ** 31:
            raise OverflowError("max_len out of range")
        return max_len, stride

    def encode_windows(self, texts, pair_texts=None, max_len=512, stride=0, token_type_ids=True, sequence_id=False, return_offsets_mapping=False):
        """Every token of long documents, as overlapping windows of max_len (HF tokenizers' return_overflowing_tokens with a
        stride).  A single's window k holds [bos] + T[k(C-stride) : k(C-stride)+C] + [eos] with T = encode(text)[1:-1] and
        C = max_len - 2; a pair keeps its first text whole in every window and windows the second with C = max_len - len(A) - 4
        (one window, its encode_batch row, when C - stride < 1).  Each window is padded as encode_batch pads a row, so window 0
        of a document equals its encode_batch(max_len=max_len) row.  Returns a BatchEncoding with the fixed-layout planes over
        the windows plus overflow_to_sample_mapping (int64 [K]: the document of each window), window_start (int32 [K]: index
        in T of its first content token) and window_off (int64 [n+1]: first window of each document).  return_offsets_mapping:
        also 'offset_mapping', int32 [K, max_len, 2], as encode_batch gives it (a token has the same offsets in every window)."""
        max_len, stride = self._window_args(max_len, stride)
        tb, to = texts if isinstance(texts, tuple) else pack_strings(texts)
        n = len(to) - 1
        flags, pbp, pop = 0, None, None
        if pair_texts is not None:
            pb, po = pair_texts if isinstance(pair_texts, tuple) else pack_strings(pair_texts)
            if len(po) - 1 != n:
                raise ValueError("texts and pair_texts differ in length")
            pb, po = np.ascontiguousarray(pb, dtype=np.uint8), np.ascontiguousarray(po, dtype=np.int64)
            pbp, pop = pb.ctypes.data, po.ctypes.data
            flags = (L.WANT_TOKEN_TYPE if token_type_ids else 0) | (L.WANT_SEQUENCE_ID if sequence_id else 0)
        if return_offsets_mapping:
            flags |= L.WANT_OFFSETS
        tb, to = np.ascontiguousarray(tb, dtype=np.uint8), np.ascontiguousarray(to, dtype=np.int64)
        w = L.Windows()
        rc = self._lib.genztok_encode_windows(self._h, tb.ctypes.data, to.ctypes.data, pbp, pop, n, max_len, stride, flags, C.byref(w))
        if rc:
            self._err(rc, "genztok_encode_windows")
        owner = _EncodedOwner(self, w, "genztok_free_windows")
        K = int(w.enc.n)
        r = self._wrap(w.enc, K, True, owner)
        r["overflow_to_sample_mapping"] = _view(w.win_doc, K, C.c_int64, np.int64, owner)
        r["window_start"] = _view(w.win_start, K, C.c_int32, np.int32, owner)
        r["window_off"] = _view(w.win_off, n + 1, C.c_int64, np.int64, owner)
        return r

    def encode_windows_device(self, d_text, d_text_off, d_pair=None, d_pair_off=None, max_len=512, stride=0, token_type_ids=True,
                              sequence_id=False, text_bytes=None, pair_bytes=None, return_offsets_mapping=False):
        """encode_windows with everything resident on the GPU: inputs as for encode_device, outputs torch tensors on the input's
        device written on torch's current stream (same keys as encode_windows; 'offset_mapping' int32 [K, max_len, 2] with
        return_offsets_mapping).  The number of windows is read back between the two steps (one synchronisation); the planes
        are then written without another.  Window 0 of each document (rows window_off[:-1]) is its encode_batch row."""
        import torch
        max_len, stride = self._window_args(max_len, stride)
        n = d_text_off.numel() - 1
        dev = d_text.device
        has_pair = d_pair_off is not None
        flags = ((L.WANT_TOKEN_TYPE if token_type_ids else 0) | (L.WANT_SEQUENCE_ID if sequence_id else 0)) if has_pair else 0
        if return_offsets_mapping:
            flags |= L.WANT_OFFSETS
        tbytes = d_text.numel() if text_bytes is None else text_bytes
        pbytes = (d_pair.numel() if pair_bytes is None else pair_bytes) if has_pair else 0
        args = (self._h, 0, d_text.data_ptr(), d_text_off.data_ptr(), tbytes, d_pair.data_ptr() if has_pair else None,
                d_pair_off.data_ptr() if has_pair else None, pbytes, n, max_len, stride, flags)
        st = self._torch_stream(dev)
        win_off = torch.empty((n + 1,), dtype=torch.int64, device=dev)
        K = C.c_int64()
        rc = self._lib.genztok_encode_windows_device(*args, win_off.data_ptr(), None, None, None, C.byref(K), st)
        if rc:
            self._err(rc, "genztok_encode_windows_device")
        K = int(K.value)
        out = {"input_ids": torch.empty((K, max_len), dtype=torch.int32, device=dev),
               "attention_mask": torch.empty((K, max_len), dtype=torch.uint8, device=dev),
               "row_len": torch.empty((K,), dtype=torch.int32, device=dev)}
        if has_pair:
            if token_type_ids:
                out["token_type_ids"] = torch.empty((K, max_len), dtype=torch.int8, device=dev)
            if sequence_id:
                out["sequence_id"] = torch.empty((K, max_len), dtype=torch.int8, device=dev)
            out["seq_len"] = torch.empty((K,), dtype=torch.int32, device=dev)
            out["row_status"] = torch.empty((K,), dtype=torch.uint8, device=dev)
        if return_offsets_mapping:
            out["offset_mapping"] = torch.empty((K, max_len, 2), dtype=torch.int32, device=dev)
        out["overflow_to_sample_mapping"] = torch.empty((K,), dtype=torch.int64, device=dev)
        out["window_start"] = torch.empty((K,), dtype=torch.int32, device=dev)
        out["window_off"] = win_off
        P = L.DevPlanes()
        for k in ("input_ids", "attention_mask", "token_type_ids", "sequence_id", "row_len", "seq_len", "row_status"):
            setattr(P, k, out[k].data_ptr() if k in out else None)
        P.offsets = out["offset_mapping"].data_ptr() if return_offsets_mapping else None
        rc = self._lib.genztok_encode_windows_device(*args, win_off.data_ptr(), C.byref(P), out["overflow_to_sample_mapping"].data_ptr(),
                                                     out["window_start"].data_ptr(), None, st)
        if rc:
            self._err(rc, "genztok_encode_windows_device")
        return out

    def decode_batch(self, ids, offsets=None):
        """Decode rows of ids: a 2-D int array (fixed width), or flat ids + int64 offsets[n+1].  Returns list[str]."""
        ids = np.asarray(ids)
        if offsets is None:
            if ids.ndim != 2:
                raise ValueError("decode_batch needs a 2-D array or (flat ids, offsets)")
            n, width = ids.shape
            flat = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1) if ids.dtype.kind in "iu" and ids.dtype.itemsize <= 4 and ids.dtype != np.uint32 \
                else self._ids_to_int32(ids.reshape(-1))
            offp = None
        else:
            offsets = np.ascontiguousarray(offsets, dtype=np.int64)
            n, width = len(offsets) - 1, 0
            flat = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1) if ids.dtype.kind in "iu" and ids.dtype.itemsize <= 4 and ids.dtype != np.uint32 \
                else self._ids_to_int32(ids.reshape(-1))                   # (an id of 2**32 + 5 is not id 5: it decodes to the unk token)
            offp = offsets.ctypes.data
        out = L.Text()
        rc = self._lib.genztok_decode(self._hd, flat.ctypes.data, offp, n, width, C.byref(out))
        if rc:
            self._err(rc, "genztok_decode")
        try:
            off = np.ctypeslib.as_array(out.off, shape=(n + 1,)).copy()
            raw = C.string_at(out.bytes, int(out.total)) if out.total else b""
        finally:
            self._lib.genztok_free_text(self._hd, C.byref(out))
        return [raw[off[i]:off[i + 1]].decode("utf-8", "surrogatepass") for i in range(n)]

    def encode_device(self, d_text, d_text_off, d_pair=None, d_pair_off=None, max_len=128, token_type_ids=True, sequence_id=False,
                      out=None, text_bytes=None, pair_bytes=None, truncation=True, bpe_dropout=None, seed=0, row_keys=None):
        """Fixed-layout encode with everything resident on the GPU.  Inputs are torch CUDA tensors (uint8 bytes whose
        storage is 16-byte aligned and int64 offsets[n+1]); outputs are torch tensors (DLPack-exportable) on the same
        device, written on torch's current stream.  Nothing crosses PCIe and the call does not synchronise.
        truncation: True (the reference cut) or a pair strategy as in encode_batch; with a strategy and pairs the call
        synchronises once per text to size the token streams, and row_status 2 marks the rows the strategy cannot truncate.
        bpe_dropout, seed, row_keys: BPE-dropout as in encode_batch.  With row_keys None or an int64 CUDA tensor [n] on the input's
        device the call does not synchronise; row_keys in host memory (a numpy array, a list, a CPU tensor) is first copied to the
        device with a blocking copy."""
        import torch
        if not isinstance(truncation, str) and not truncation:
            raise ValueError("encode_device always truncates (the fixed layout): truncation must be True or a strategy name")
        drop = None
        if bpe_dropout is not None:
            drop = _dropout_args(bpe_dropout, seed, max_len, True, truncation)
            strategy = 0
        else:
            strategy = _strategy_flag(truncation, max_len)
        n = d_text_off.numel() - 1
        dev = d_text.device
        keys = None
        if drop is not None and row_keys is not None:
            keys = row_keys if isinstance(row_keys, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(row_keys, dtype=np.int64)))
            if tuple(keys.shape) != (n,):
                raise ValueError("row_keys must have shape (%d,) (got %s)" % (n, tuple(keys.shape)))
            keys = keys.to(dev, torch.int64).contiguous()
        has_pair = d_pair_off is not None
        if out is None:
            out = {"input_ids": torch.empty((n, max_len), dtype=torch.int32, device=dev),
                   "attention_mask": torch.empty((n, max_len), dtype=torch.uint8, device=dev),
                   "row_len": torch.empty((n,), dtype=torch.int32, device=dev)}
            if has_pair:
                if token_type_ids:
                    out["token_type_ids"] = torch.empty((n, max_len), dtype=torch.int8, device=dev)
                if sequence_id:
                    out["sequence_id"] = torch.empty((n, max_len), dtype=torch.int8, device=dev)
                out["seq_len"] = torch.empty((n,), dtype=torch.int32, device=dev)
                out["row_status"] = torch.empty((n,), dtype=torch.uint8, device=dev)
        P = L.DevPlanes()
        for k in ("input_ids", "attention_mask", "token_type_ids", "sequence_id", "row_len", "seq_len", "row_status"):
            setattr(P, k, out[k].data_ptr() if k in out else None)
        flags = strategy
        if has_pair:
            flags |= (L.WANT_TOKEN_TYPE if "token_type_ids" in out else 0) | (L.WANT_SEQUENCE_ID if "sequence_id" in out else 0)
        tbytes = d_text.numel() if text_bytes is None else text_bytes
        pbytes = (d_pair.numel() if pair_bytes is None else pair_bytes) if has_pair else 0
        slot = 0
        if drop is not None:
            rc = self._lib.genztok_encode_dropout_device(self._h, slot, d_text.data_ptr(), d_text_off.data_ptr(), tbytes,
                                                         d_pair.data_ptr() if has_pair else None, d_pair_off.data_ptr() if has_pair else None,
                                                         pbytes, n, int(max_len), flags, drop[0], drop[1], keys.data_ptr() if keys is not None else None,
                                                         C.byref(P), self._torch_stream(dev))
            if rc:
                self._err(rc, "genztok_encode_dropout_device")
            return out
        rc = self._lib.genztok_encode_device(self._h, slot, d_text.data_ptr(), d_text_off.data_ptr(), tbytes,
                                             d_pair.data_ptr() if has_pair else None, d_pair_off.data_ptr() if has_pair else None, pbytes,
                                             n, int(max_len), flags, C.byref(P), self._torch_stream(dev))
        if rc:
            self._err(rc, "genztok_encode_device")
        return out

    @staticmethod
    def _torch_stream(dev):
        """torch's current stream as a cudaStream_t; its default stream (handle 0) is the legacy stream, (cudaStream_t)1,
        because the C ABI reads NULL as "the handle's own stream"."""
        import torch
        return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream or 1)

    def decode_device(self, d_ids, d_ids_off=None, out=None, sync=True):
        """Decode rows resident on the GPU: 2-D int32 tensor, or flat int32 + int64 offsets.  Returns (uint8 bytes, int64 offsets) tensors.
        `out`: a uint8 CUDA tensor to write the text into (a reused ring for streamed batches): sizes and text are then produced
        without a host read in between, and the returned bytes are a view of it; when the text does not fit, a tensor of the
        right size is allocated and returned instead.  `sync=False` (with `out`) returns (out, offsets) without waiting for the
        device: the text is out[:offsets[-1]] and nothing is written if it does not fit."""
        import torch
        dev = d_ids.device
        if d_ids_off is None:
            n, width = d_ids.shape
            offp = None
        else:
            n, width = d_ids_off.numel() - 1, 0
            offp = d_ids_off.data_ptr()
        out_off = torch.empty((n + 1,), dtype=torch.int64, device=dev)
        total = C.c_int64()
        st = self._torch_stream(dev)
        if out is not None and out.device == dev and out.dtype == torch.uint8 and out.data_ptr() % 16 == 0 and out.numel() > 0:
            rc = self._lib.genztok_decode_device_into(self._hd, 0, d_ids.data_ptr(), offp, n, width, out_off.data_ptr(), out.data_ptr(), out.numel(),
                                                      C.byref(total) if sync else None, st)
            if rc:
                self._err(rc, "genztok_decode_device_into")
            if not sync:
                return out, out_off
            if total.value <= out.numel():
                return out[:total.value], out_off
        else:
            if not sync:
                raise ValueError("decode_device(sync=False) needs a uint8 CUDA tensor `out` (16-byte aligned) to write into")
            rc = self._lib.genztok_decode_device(self._hd, 0, d_ids.data_ptr(), offp, n, width, out_off.data_ptr(), None, C.byref(total), st)
            if rc:
                self._err(rc, "genztok_decode_device")
        out = torch.empty((max(total.value, 1),), dtype=torch.uint8, device=dev)
        rc = self._lib.genztok_decode_device(self._hd, 0, d_ids.data_ptr(), offp, n, width, out_off.data_ptr(), out.data_ptr(), None, st)
        if rc:
            self._err(rc, "genztok_decode_device")
        return out[:total.value], out_off

    # ---- extractive question answering over the windows' planes ------------------------------------------------------------
    def _qa_planes(self, enc):
        """(torch offsets [K, W, 2], window_off [n + 1], has_pair, device, host_form) of an encode_windows(_device) result or a
        fixed-layout encode_batch result with offsets (one window per document), on the handle's device."""
        import torch
        if "offset_mapping" not in enc:
            raise ValueError("qa: the encoding has no 'offset_mapping'; encode with return_offsets_mapping=True")
        om = enc["offset_mapping"]
        if om.ndim != 3 or om.shape[2] != 2:
            raise ValueError("qa: 'offset_mapping' must be the fixed [windows, max_len, 2] layout (got shape %s; ragged results "
                             "are not supported)" % (tuple(om.shape),))
        K, W = int(om.shape[0]), int(om.shape[1])
        if W < 3:
            raise ValueError("qa: max_len >= 3 needed (got %d)" % W)
        host = not isinstance(om, torch.Tensor)
        if host:
            if not self._device_ids:
                raise GenztokError("qa: this handle was created without a CUDA device; there is no CPU path")
            dev = torch.device("cuda", self._device_ids[0])
            om = torch.from_numpy(np.ascontiguousarray(om, dtype=np.int32)).to(dev)
        else:
            dev = om.device
            om = om.to(torch.int32).contiguous()
        wo = enc.get("window_off")
        if wo is None:
            wo = torch.arange(K + 1, dtype=torch.int64, device=dev)
        else:
            wo = (torch.from_numpy(np.ascontiguousarray(wo, dtype=np.int64)) if not isinstance(wo, torch.Tensor) else wo).to(dev, torch.int64).contiguous()
            if wo.ndim != 1 or wo.numel() < 1:
                raise ValueError("qa: 'window_off' must be int64 [n + 1]")
        return om, wo, "seq_len" in enc, dev, host

    @staticmethod
    def _qa_rows(x, shape, dtype, dev, what):
        import torch
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(x)))
        if tuple(t.shape) != tuple(shape):
            raise ValueError("qa: %s must have shape %s (got %s)" % (what, tuple(shape), tuple(t.shape)))
        return t.to(dev, dtype).contiguous()

    def qa_labels(self, enc, answers, unit="byte", context=None):
        """Extractive-QA training labels: (start_positions, end_positions), int64 [K], one pair per window.
        `enc`: an encode_windows / encode_windows_device result, or a fixed-layout encode_batch result (one window per
        document), made with return_offsets_mapping=True.  `answers`: [n, 2] spans [a0, a1) in the windowed text (`texts[d]`,
        or `pair_texts[d]` for pairs), in bytes of its UTF-8 ('surrogatepass') form with unit="byte", in Python str indices
        with unit="char" -- then `context` is that text: list[str], packed (bytes, offsets) or CUDA tensors (d_text 16-byte
        aligned, d_text_off).  A window's context columns come from the offsets alone (singles: end > 0; pairs: end > 0
        after the first (0, 0) column >= 1); its label is (first, last) of the context columns that overlap the answer when
        they hold all of it, else (0, 0).  No answer (a1 <= a0) and spans past the end give (0, 0).  Device results stay on
        their device on torch's current stream; numpy results are copied to the handle's device (8 bytes per column of
        offsets) and the labels back."""
        import torch
        if unit not in ("byte", "char"):
            raise ValueError("qa_labels: unit must be 'byte' or 'char' (got %r)" % (unit,))
        om, wo, has_pair, dev, host = self._qa_planes(enc)
        K, W = int(om.shape[0]), int(om.shape[1])
        n = wo.numel() - 1
        ans = self._qa_rows(answers, (n, 2), torch.int64, dev, "answers")
        tx = toff = None
        nb = 0
        if unit == "char":
            if context is None:
                raise ValueError("qa_labels: unit='char' needs `context`, the windowed text")
            if isinstance(context, tuple) and isinstance(context[0], torch.Tensor):
                tx, toff = context[0], context[1].to(dev, torch.int64).contiguous()
                nb = tx.numel()
            else:
                b, o = context if isinstance(context, tuple) else pack_strings(context)
                b = np.ascontiguousarray(b, dtype=np.uint8)
                nb = len(b)
                tx = torch.from_numpy(np.concatenate([b, np.zeros((-nb) % 16 + 16, dtype=np.uint8)])).to(dev)
                toff = torch.from_numpy(np.ascontiguousarray(o, dtype=np.int64)).to(dev)
            if toff.numel() != n + 1:
                raise ValueError("qa_labels: `context` holds %d documents, the encoding %d" % (toff.numel() - 1, n))
        start = torch.empty((K,), dtype=torch.int64, device=dev)
        end = torch.empty((K,), dtype=torch.int64, device=dev)
        rc = self._lib.genztok_qa_labels_device(self._h, 0, om.data_ptr(), K, W, int(has_pair), wo.data_ptr(), n, ans.data_ptr(),
                                                L.QA_CHARS if unit == "char" else L.QA_BYTES, tx.data_ptr() if tx is not None else None,
                                                toff.data_ptr() if toff is not None else None, nb, start.data_ptr(), end.data_ptr(), self._torch_stream(dev))
        if rc:
            self._err(rc, "genztok_qa_labels_device")
        if host:
            return start.cpu().numpy(), end.cpu().numpy()
        return start, end

    def qa_best_spans(self, enc, start_logits, end_logits, max_answer_len=30):
        """The best answer span per document from a QA model's start / end logits ([K, W], one row per window of `enc`, as
        for qa_labels; not float32 is converted with .float()).  Candidates are (window i of the document, s, e) with s <= e
        context columns of i and e - s + 1 <= max_answer_len, scored start_logits[i, s] + end_logits[i, e] (one float32 add);
        the best is the largest score, ties to the smallest i, then s, then e, and a NaN score is never taken.  This is the
        exact maximum over every valid pair (HF's top-20 x top-20 pre-filter can only find a lower or equal one).  Returns a
        dict with, per document: 'score' (float32), 'null_score' (min over its windows of start_logits[i, 0] + end_logits[i, 0],
        SQuAD v2's no-answer score), 'window' (int64 global window, -1 with no candidate), 'columns' (int32 [n, 2] (s, e)) and
        'span' (int32 [n, 2], the answer's byte range in the document); a document without a candidate gets score -inf and
        (0, 0).  Device results stay on their device; numpy results are copied to the handle's device and back."""
        import torch
        max_answer_len = operator.index(max_answer_len)
        if max_answer_len < 1:
            raise ValueError("qa_best_spans: max_answer_len >= 1 needed (got %d)" % max_answer_len)
        om, wo, has_pair, dev, host = self._qa_planes(enc)
        K, W = int(om.shape[0]), int(om.shape[1])
        n = wo.numel() - 1
        sl = self._qa_rows(start_logits if isinstance(start_logits, torch.Tensor) else np.asarray(start_logits, dtype=np.float32), (K, W), torch.float32, dev, "start_logits")
        el = self._qa_rows(end_logits if isinstance(end_logits, torch.Tensor) else np.asarray(end_logits, dtype=np.float32), (K, W), torch.float32, dev, "end_logits")
        out = {"score": torch.empty((n,), dtype=torch.float32, device=dev), "null_score": torch.empty((n,), dtype=torch.float32, device=dev),
               "window": torch.empty((n,), dtype=torch.int64, device=dev), "columns": torch.empty((n, 2), dtype=torch.int32, device=dev),
               "span": torch.empty((n, 2), dtype=torch.int32, device=dev)}
        rc = self._lib.genztok_qa_best_spans_device(self._h, 0, sl.data_ptr(), el.data_ptr(), om.data_ptr(), K, W, int(has_pair), wo.data_ptr(), n,
                                                    min(max_answer_len, 2 ** 31 - 1), out["score"].data_ptr(), out["null_score"].data_ptr(),
                                                    out["window"].data_ptr(), out["columns"].data_ptr(), out["span"].data_ptr(), self._torch_stream(dev))
        if rc:
            self._err(rc, "genztok_qa_best_spans_device")
        if host:
            return {k: v.cpu().numpy() for k, v in out.items()}
        return out

    # ---- masked language modelling ---------------------------------------------------------------------------------------------
    def mlm_mask(self, input_ids, seed, mlm_probability=0.15, whole_word=False, mask_replace_prob=0.8, random_replace_prob=0.1, row_keys=None):
        """Masked-language-model inputs and labels from a fixed-layout id plane [n, W] (an encode_batch, encode_device,
        encode_windows(_device) or DataCollection batch's input_ids): returns (masked_ids int32 [n, W], labels int64 [n, W]).
        Eligible columns (ids in [0, n_ids) that are not special) are selected with probability `mlm_probability`, per token or,
        with `whole_word`, per word (a piece whose vocab string ends in "@@" continues into the next column); a selected column
        becomes the mask id with probability `mask_replace_prob`, a random non-special vocab id with `random_replace_prob`,
        else keeps its id, and is labelled with its original id; every other column keeps its id and is labelled -100.  The
        draws are a pure function of (seed, row key, row contents), row r's key being `row_keys[r]` (int64 [n]) or r: take a
        new `seed` per epoch for dynamic masking.  include/genztok.h states the hashes.  A CUDA tensor stays on its device, on
        torch's current stream; a numpy plane is copied to the handle's device and the results back.  Other integer dtypes are
        converted to int32, ids outside the int32 range becoming -1 or 2^31 - 1 (ineligible either way, and so returned);
        float, bool and complex planes raise TypeError."""
        import torch
        host = not isinstance(input_ids, torch.Tensor)
        if host:
            a = np.asarray(input_ids)
            if a.dtype.kind not in "iu":
                raise TypeError("mlm_mask: input_ids must hold integers (got %s)" % a.dtype)
            if not self._device_ids:
                raise GenztokError("mlm_mask: this handle was created without a CUDA device; there is no CPU path")
            dev = torch.device("cuda", self._device_ids[0])
            if a.dtype.itemsize >= 4 and a.dtype != np.int32:                # ids outside int32 can never be eligible: keep them so
                a = np.minimum(a, 2 ** 31 - 1) if a.dtype.kind == "u" else np.clip(a, -1, 2 ** 31 - 1)
            ids = torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
        else:
            dev = input_ids.device
            if input_ids.dtype not in (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8):
                raise TypeError("mlm_mask: input_ids must hold integers (got %s)" % input_ids.dtype)
            ids = input_ids
            if ids.dtype == torch.int64:                                    # ids outside int32 can never be eligible: keep them so
                ids = ids.clamp(-1, 2 ** 31 - 1)
            ids = ids.to(torch.int32).contiguous()
        if ids.ndim != 2:
            raise ValueError("mlm_mask: input_ids must be a fixed-layout [n, W] plane (got shape %s)" % (tuple(ids.shape),))
        n, W = int(ids.shape[0]), int(ids.shape[1])
        keys = None
        if row_keys is not None:
            keys = row_keys if isinstance(row_keys, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(row_keys, dtype=np.int64)))
            if tuple(keys.shape) != (n,):
                raise ValueError("mlm_mask: row_keys must have shape (%d,) (got %s)" % (n, tuple(keys.shape)))
            keys = keys.to(dev, torch.int64).contiguous()
        out = torch.empty((n, W), dtype=torch.int32, device=dev)
        labels = torch.empty((n, W), dtype=torch.int64, device=dev)
        rc = self._lib.genztok_mlm_mask_device(self._h, 0, ids.data_ptr(), n, W, keys.data_ptr() if keys is not None else None,
                                               operator.index(seed) & (2 ** 64 - 1), float(mlm_probability), float(mask_replace_prob),
                                               float(random_replace_prob), int(bool(whole_word)), out.data_ptr(), labels.data_ptr(),
                                               self._torch_stream(dev))
        if rc:
            self._err(rc, "genztok_mlm_mask_device")
        if host:
            return out.cpu().numpy(), labels.cpu().numpy()
        return out, labels

    # ---- measurement plumbing (bench.py, tests): synthetic workload on the device, plane digest, error counter -----------
    def synth_device(self, seed, doc0, n, side=0, lo=3, hi=13, noise=0.0, device=None):
        """Documents [doc0, doc0 + n) of workload.generate_hashed produced on the GPU: (uint8 bytes padded for 16-byte loads,
        int64 offsets[n+1], byte count)."""
        import torch
        from . import workload
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        if not getattr(self, "_synth_ready", False):
            T = workload.default_synth_tables()
            keep = [np.ascontiguousarray(a) for a in (T.wblob, T.wstart, T.wlen, T.cdf32, T.eblob, T.estart, T.elen)]
            rc = self._lib.genztok_synth_init(self._h, 0, keep[0].ctypes.data, len(keep[0]), keep[1].ctypes.data, keep[2].ctypes.data, keep[3].ctypes.data, T.nw,
                                              keep[4].ctypes.data, len(keep[4]), keep[5].ctypes.data, keep[6].ctypes.data, T.ne)
            if rc:
                self._err(rc, "genztok_synth_init")
            self._synth_ready = True
        st = self._torch_stream(dev)
        off = torch.empty((n + 1,), dtype=torch.int64, device=dev)
        total = C.c_int64()
        thr = workload.noise_threshold(noise)
        rc = self._lib.genztok_synth_device(self._h, 0, int(seed), int(doc0), int(n), int(side), int(lo), int(hi), thr, off.data_ptr(), None, C.byref(total), st)
        if rc:
            self._err(rc, "genztok_synth_device")
        nb = int(total.value)
        data = torch.zeros((nb + (-nb) % 16 + 32,), dtype=torch.uint8, device=dev)
        rc = self._lib.genztok_synth_device(self._h, 0, int(seed), int(doc0), int(n), int(side), int(lo), int(hi), thr, off.data_ptr(), data.data_ptr(), None, st)
        if rc:
            self._err(rc, "genztok_synth_device")
        return data, off, nb

    def digest_device(self, planes, row0, acc):
        """acc (1-element int64 CUDA tensor) += order-independent digest of the [n, W] planes whose first row is global row `row0`."""
        ids = planes["input_ids"]
        n, W = ids.shape
        tt = planes.get("token_type_ids")
        rc = self._lib.genztok_digest_device(self._h, 0, ids.data_ptr(), planes["attention_mask"].data_ptr(), tt.data_ptr() if tt is not None else None,
                                             int(n), int(W), int(row0), acc.data_ptr(), self._torch_stream(ids.device))
        if rc:
            self._err(rc, "genztok_digest_device")

    def check_errors(self, device=None):
        """Raises if the device pipeline counted an inconsistency (the asynchronous device path cannot report them itself)."""
        import torch
        n = C.c_int64()
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        rc = self._lib.genztok_check_errors(self._h, 0, self._torch_stream(dev), C.byref(n))
        if rc:
            self._err(rc, "genztok_check_errors")
        return int(n.value)

    # ---- engine introspection ----------------------------------------------------------------------------
    def launch_count(self):
        return int(self._lib.genztok_launch_count(self._h))

    def set_profiling(self, on):
        self._lib.genztok_set_profiling(self._h, int(bool(on)))

    def profile_report(self, reset=True):
        import json
        n = self._lib.genztok_profile_report(self._h, None, 0, 0)
        buf = C.create_string_buffer(int(n) + 16)
        self._lib.genztok_profile_report(self._h, buf, len(buf), int(bool(reset)))
        return json.loads(buf.value.decode())

    def cache_reset(self):
        rc = self._lib.genztok_cache_reset(self._h)
        if rc:
            self._err(rc, "genztok_cache_reset")

    @classmethod
    def fromFile(cls, vocab_file, bpe_file, **kw):
        """tokenize.py:261-267: custom files, default special-token strings."""
        tokenize = cls.__new__(cls)
        tokenize.vocab_file = vocab_file
        tokenize.bpe_file = bpe_file
        tokenize.__init__(**kw)
        return tokenize
