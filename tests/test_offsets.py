"""offset_mapping: each token's [start, end) byte range in its own document (HF tokenizers' return_offsets_mapping).

The expected offsets come from the oracle and Python alone: words are re.finditer(r"\\S+\\n?") over the str, their byte positions
are 'surrogatepass' UTF-8 lengths, their pieces are oracle.bpe(word) (pieces joined by spaces, "@@" closing every piece but the
last), and every token that is not from the text -- <s>, </s>, pads, the </s> truncation forces -- is (0, 0).  The framed lists
are then cut as tokenize.py:141-146 cut the ids, and windows as tests/test_windows.py cuts them.  Argument checks and the
host-only handle run on the CPU; everything else on the GPU."""
import ctypes as C
import re

import numpy as np
import pytest

from genz_tokenize_b200 import _lib as L

gpu = pytest.mark.gpu
WORD = re.compile(r"\S+\n?")
ZERO = (0, 0)


def blen(s):
    return len(s.encode("utf-8", "surrogatepass"))


def word_offsets(oracle, s):
    """Offsets of the tokens of encode(s)[1:-1], word by word."""
    out = []
    for m in WORD.finditer(s):
        w = m.group(0)
        a = blen(s[:m.start()])
        pieces = oracle.bpe(w).split(" ")
        texts = []
        for k, p in enumerate(pieces):
            if k < len(pieces) - 1:
                assert p.endswith("@@"), (w, pieces)
                p = p[:-2]
            elif p.endswith("</w>"):
                p = p[:-4]
            texts.append(p)
        assert "".join(texts) == w, (w, pieces)                       # the pieces tile the word
        for p in texts:
            out.append((a, a + blen(p)))
            a += blen(p)
    return out


def framed_offsets(oracle, s, p=None):
    """The offsets of the reference's full row: [<s>] A [</s>] or [<s>] A [</s> </s>] B [</s>]."""
    A = word_offsets(oracle, s)
    if p is None:
        return [ZERO] + A + [ZERO]
    return [ZERO] + A + [ZERO, ZERO] + word_offsets(oracle, p) + [ZERO]


def py_head(n, k):
    return max(n + k, 0) if k < 0 else min(k, n)


def cut_row(F, max_len, padding, truncation):
    """tokenize.py:141-146 (__padding) on the offsets list."""
    if max_len is not None and padding:
        if len(F) < max_len:
            return F + [ZERO] * (max_len - len(F))
        if truncation:
            return F[:py_head(len(F), max_len - 1)] + [ZERO]
    return F


def expected(oracle, texts, pairs, max_len, padding, truncation):
    rows = [cut_row(framed_offsets(oracle, t, None if pairs is None else pairs[i]), max_len, padding, truncation) for i, t in enumerate(texts)]
    return rows


def rows_of(r, n):
    """The offset_mapping of an encode_batch result as a list of per-row lists."""
    om = r["offset_mapping"]
    if om.ndim == 3:
        return [[tuple(x) for x in om[i].tolist()] for i in range(n)]
    off = r["row_off"]
    return [[tuple(x) for x in om[off[i]:off[i + 1]].tolist()] for i in range(n)]


def assert_same_other_outputs(a, b, what):
    """Every output but offset_mapping is the same with and without offsets."""
    ka, kb = set(a) - {"offset_mapping"}, set(b)
    assert ka == kb, (what, ka ^ kb)
    for k in ka:
        x, y = a[k], b[k]
        if isinstance(x, np.ndarray):
            assert x.shape == y.shape and x.dtype == y.dtype and np.array_equal(x, y), (what, k)
        else:
            assert x == y, (what, k)


# ---- CPU ----------------------------------------------------------------------------------------------------------------------
def test_word_offsets_tile_the_text(oracle):
    # the helper the GPU tests rest on, on the oracle alone
    s = "xin chào\u00a0sinh_viên\n\n</s> \U0001F600x  \ud800ab @@ </w>\tđ\u2028z"
    F = word_offsets(oracle, s)
    b = s.encode("utf-8", "surrogatepass")
    words = [m.group(0).encode("utf-8", "surrogatepass") for m in WORD.finditer(s)]
    assert b"".join(b[x:y] for x, y in F) == b"".join(words)
    assert all(y > x for x, y in F)
    r = oracle.encode_batch([s], None)
    assert len(F) + 2 == len(r["ids"])


def test_offsets_flag_rejected_by_encode_device_and_host_only_handle():
    from genz_tokenize_b200 import Tokenize
    from genz_tokenize_b200.tokenizer import GenztokError
    t = Tokenize(devices=[])
    lib = L.load()
    P = L.DevPlanes()
    z = np.zeros(64, dtype=np.uint8)
    o = np.array([0, 3], dtype=np.int64)
    assert lib.genztok_encode_device(t._h, 0, z.ctypes.data, o.ctypes.data, 3, None, None, 0, 1, 16, L.WANT_OFFSETS, C.byref(P), None) == L.E_INVALID
    assert b"offsets" in lib.genztok_last_error(t._h)
    e = L.Encoded()
    assert lib.genztok_encode(t._h, z.ctypes.data, o.ctypes.data, None, None, 1, 16, 1, 1, L.WANT_OFFSETS, C.byref(e)) == L.E_NODEVICE
    w = L.Windows()
    assert lib.genztok_encode_windows(t._h, z.ctypes.data, o.ctypes.data, None, None, 1, 16, 2, L.WANT_OFFSETS, C.byref(w)) == L.E_NODEVICE
    with pytest.raises(GenztokError, match="no CPU path"):
        t.encode_batch(["xin chào"], max_len=16, return_offsets_mapping=True)
    with pytest.raises(GenztokError, match="no CPU path"):
        t.encode_windows(["xin chào"], max_len=16, stride=2, return_offsets_mapping=True)


def test_abi_mirrors():
    # genztok_encoded_t / genztok_dev_planes_t end with the offsets pointer; genztok_windows_t embeds the former
    assert L.Encoded._fields_[-1][0] == "offsets" and L.DevPlanes._fields_[-1][0] == "offsets"
    assert L.Windows.win_off.offset == C.sizeof(L.Encoded) + 8
    assert L.WANT_OFFSETS == 8


# ---- GPU ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tok():
    from genz_tokenize_b200 import Tokenize
    return Tokenize(devices=[0])


WS = "\t\n\x0b\x0c\r\x1c\x1d\x1e\x1f \x85\xa0\u1680\u2000\u2001\u2002\u2003\u2004\u2005\u2006\u2007\u2008\u2009\u200a\u2028\u2029\u202f\u205f\u3000"


def unpack(packed):
    """(uint8 bytes, int64 offsets[n+1]) -> list[str]"""
    b, o = packed
    return [bytes(b[o[i]:o[i + 1]]).decode("utf-8", "surrogatepass") for i in range(len(o) - 1)]


def noisy_rows(seed, n):
    """Rows with every kind of word the offsets must get right."""
    from genz_tokenize_b200 import workload
    assert len(WS) == 29
    rng = np.random.default_rng(seed)
    base = unpack(workload.generate(seed, n, 0, 40, 0.05))
    specials = ["</s>", "</w>", "@@", "<s>", "<pad>", "\U0001F600", "\U0001F600x\U00010348", "\ud800", "a\udfffb", "đường", "x" * 1200,
                "sinh_viên" * 150, "ab" * 600 + "\U0001F600", "1"]
    out = []
    for s in base:
        words = s.split(" ") if s else []
        for _ in range(int(rng.integers(0, 4))):
            words.insert(int(rng.integers(0, len(words) + 1)), specials[int(rng.integers(0, len(specials)))])
        seps = [WS[int(rng.integers(0, len(WS)))] * int(rng.integers(1, 3)) for _ in words]
        t = "".join(w + sp for w, sp in zip(words, seps))
        if rng.random() < 0.3:
            t = WS[int(rng.integers(0, len(WS)))] + t
        out.append(t)
    return out


README = ("sinh_viên công_nghệ", "hello")


@gpu
def test_readme_vector(tok, oracle):
    got = tok(README[0], return_offsets_mapping=True)
    assert got["offset_mapping"] == [ZERO, (0, 10), (11, 23), ZERO]
    got = tok(README[0], README[1], max_len=10, return_offsets_mapping=True)
    assert got["input_ids"] == [1, 770, 1444, 2, 2, 30469, 2, 0, 0, 0]
    assert got["offset_mapping"] == [ZERO, (0, 10), (11, 23), ZERO, ZERO, (0, 5), ZERO, ZERO, ZERO, ZERO]
    assert got["offset_mapping"] == cut_row(framed_offsets(oracle, *README), 10, True, True)
    plain = tok(README[0], README[1], max_len=10)
    assert {k: v for k, v in got.items() if k != "offset_mapping"} == plain


REGIMES = [dict(max_len=None), dict(max_len=16, padding=False), dict(max_len=1), dict(max_len=2), dict(max_len=3), dict(max_len=16),
           dict(max_len=256), dict(max_len=16, truncation=False), dict(max_len=0), dict(max_len=-1), dict(max_len=16, return_offset=True),
           dict(max_len=None, return_offset=True)]


@gpu
@pytest.mark.parametrize("kw", REGIMES, ids=[str(sorted(k.items())) for k in REGIMES])
def test_offsets_match_oracle_every_regime(tok, oracle, kw):
    texts, pairs = noisy_rows(1, 400), noisy_rows(2, 400)
    ml = kw.get("max_len")
    for p in (None, pairs):
        r = tok.encode_batch(texts, p, return_offsets_mapping=True, **kw)
        plain = tok.encode_batch(texts, p, **kw)
        what = "%s pairs=%s" % (kw, p is not None)
        assert_same_other_outputs(r, plain, what)
        fixed = ml is not None and ml >= 1 and kw.get("padding", True) and kw.get("truncation", True) and not kw.get("return_offset")
        assert r["offset_mapping"].dtype == np.int32
        assert r["offset_mapping"].shape == ((len(texts), ml, 2) if fixed else (len(r["input_ids"]), 2)), what
        exp = expected(oracle, texts, p, ml, kw.get("padding", True), kw.get("truncation", True))
        got = rows_of(r, len(texts))
        for i in range(len(texts)):
            assert got[i] == exp[i], "%s row %d:\n ours=%s\n ref =%s\n text=%r" % (what, i, got[i][:40], exp[i][:40], texts[i][:200])
        # the row form of __call__ / BatchEncoding.row
        for i in (0, 7):
            try:
                row = r.row(i)
            except ValueError:
                continue
            assert row["offset_mapping"] == exp[i]


@gpu
def test_offsets_invariant_words_are_tiled(tok):
    texts = noisy_rows(5, 300)
    r = tok.encode_batch(texts, return_offsets_mapping=True)
    for i, s in enumerate(texts):
        b = s.encode("utf-8", "surrogatepass")
        om = r["offset_mapping"][r["row_off"][i]:r["row_off"][i + 1]]
        real = [(x, y) for x, y in om.tolist() if (x, y) != ZERO]
        assert all(y > x for x, y in real)
        assert b"".join(b[x:y] for x, y in real) == b"".join(m.group(0).encode("utf-8", "surrogatepass") for m in WORD.finditer(s))


@gpu
def test_offsets_fixed_regime_equals_flat_pipeline(tok):
    # a batch large enough that the fixed layout without offsets takes the byte-parallel pipeline
    from genz_tokenize_b200 import workload
    n = 1 << 15
    ta, tb = workload.generate_hashed(77, 0, n, 0, 3, 13, 0.01), workload.generate_hashed(77, 0, n, 1, 3, 13, 0.01)   # packed form
    for W in (64, 128):
        a = tok.encode_batch(ta, tb, max_len=W, return_offsets_mapping=True)
        b = tok.encode_batch(ta, tb, max_len=W)
        assert_same_other_outputs(a, b, "flat W=%d" % W)
        assert a["offset_mapping"].shape == (n, W, 2)


@gpu
def test_offsets_cache_states(oracle):
    # words cached by calls without offsets get their lengths later: the first-use reset, and after cache_reset
    from genz_tokenize_b200 import Tokenize
    t = Tokenize(devices=[0])
    texts = noisy_rows(9, 300)
    t.encode_batch(texts, max_len=64)
    t.encode_batch(texts)
    exp = expected(oracle, texts, None, None, True, True)
    assert rows_of(t.encode_batch(texts, return_offsets_mapping=True), len(texts)) == exp
    assert rows_of(t.encode_batch(texts, return_offsets_mapping=True), len(texts)) == exp      # now from a warm cache
    t.encode_batch(noisy_rows(10, 300), max_len=32)                                           # new words, lengths recorded
    t.cache_reset()
    assert rows_of(t.encode_batch(texts, return_offsets_mapping=True), len(texts)) == exp


@gpu
def test_offsets_chunks_and_devices(oracle):
    import torch
    from genz_tokenize_b200 import Tokenize
    texts, pairs = noisy_rows(11, 500), noisy_rows(12, 500)
    base, small = Tokenize(devices=[0]), Tokenize(devices=[0])
    small.set_option("chunk_rows", 7)
    for kw in (dict(max_len=32), dict(max_len=None)):
        x, y = base.encode_batch(texts, pairs, return_offsets_mapping=True, **kw), small.encode_batch(texts, pairs, return_offsets_mapping=True, **kw)
        assert np.array_equal(x["offset_mapping"], y["offset_mapping"])
        assert rows_of(x, len(texts)) == expected(oracle, texts, pairs, kw["max_len"], True, True)
    w0 = base.encode_windows(texts, pairs, max_len=48, stride=8, return_offsets_mapping=True)
    w1 = small.encode_windows(texts, pairs, max_len=48, stride=8, return_offsets_mapping=True)
    assert np.array_equal(w0["offset_mapping"], w1["offset_mapping"])
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    multi = Tokenize(devices=list(range(ndev)))
    for kw in (dict(max_len=32), dict(max_len=None)):
        x, y = base.encode_batch(texts, pairs, return_offsets_mapping=True, **kw), multi.encode_batch(texts, pairs, return_offsets_mapping=True, **kw)
        assert np.array_equal(x["offset_mapping"], y["offset_mapping"])
    w2 = multi.encode_windows(texts, pairs, max_len=48, stride=8, return_offsets_mapping=True)
    assert np.array_equal(w0["offset_mapping"], w2["offset_mapping"])


# ---- windows ------------------------------------------------------------------------------------------------------------------
def expected_window_offsets(oracle, texts, pairs, W, s):
    """[K, W, 2] cut from the framed offsets as test_windows.expected_windows cuts the ids."""
    from test_windows import window_count
    rows = []
    for d, t in enumerate(texts):
        A = word_offsets(oracle, t)
        if pairs is None:
            T, C_ = A, W - 2
            for k in range(window_count(len(T), W, s)):
                st = k * (C_ - s)
                rows.append([ZERO] + T[st:st + C_] + [ZERO])
        else:
            T = word_offsets(oracle, pairs[d])
            C_ = W - len(A) - 4
            for k in range(window_count(len(T), W, s, len(A))):
                st = 0 if C_ - s < 1 else k * (C_ - s)
                part = T if C_ - s < 1 else T[st:st + C_]
                rows.append([ZERO] + A + [ZERO, ZERO] + part + [ZERO])
    out = np.zeros((len(rows), W, 2), dtype=np.int32)
    for i, r in enumerate(rows):
        r = r + [ZERO] * (W - len(r)) if len(r) < W else r[:W - 1] + [ZERO]
        out[i] = np.array(r, dtype=np.int32).reshape(W, 2)
    return out


def assert_window_offsets(got, exp, what):
    assert got.shape == exp.shape, (what, got.shape, exp.shape)
    bad = np.argwhere((got != exp).any(axis=2))
    assert not len(bad), "%s: window %d column %d: ours=%s ref=%s" % (what, bad[0][0], bad[0][1], got[bad[0][0]].tolist()[:20], exp[bad[0][0]].tolist()[:20])


@gpu
@pytest.mark.parametrize("W", [3, 16, 130, 512])
def test_window_offsets_singles(tok, oracle, W):
    texts = noisy_rows(20 + W, 200)
    for s in sorted({0, min(1, W - 3), W - 3}):
        w = tok.encode_windows(texts, max_len=W, stride=s, return_offsets_mapping=True)
        plain = tok.encode_windows(texts, max_len=W, stride=s)
        assert_same_other_outputs(w, plain, "W=%d s=%d" % (W, s))
        assert_window_offsets(w["offset_mapping"], expected_window_offsets(oracle, texts, None, W, s), "singles W=%d s=%d" % (W, s))
        assert w.row(0)["offset_mapping"] == [tuple(x) for x in w["offset_mapping"][0].tolist()]


@gpu
def test_window_offsets_pairs(tok, oracle):
    from genz_tokenize_b200 import workload
    q = noisy_rows(31, 48)
    ctx = unpack(workload.long_documents(workload.default_wordlist().words, 48, lo=300, hi=2500, seed=9))
    ctx = [c + WS[i % 29] + noisy_rows(32 + i, 1)[0] for i, c in enumerate(ctx)]
    for W, s in ((384, 128), (130, 0), (16, 4)):                       # (16, 4): most questions leave no room to step
        w = tok.encode_windows(q, ctx, max_len=W, stride=s, sequence_id=True, return_offsets_mapping=True)
        assert_same_other_outputs(w, tok.encode_windows(q, ctx, max_len=W, stride=s, sequence_id=True), "pairs W=%d" % W)
        assert_window_offsets(w["offset_mapping"], expected_window_offsets(oracle, q, ctx, W, s), "pairs W=%d s=%d" % (W, s))
        # window 0 of each document is its encode_batch row, offsets included
        r = tok.encode_batch(q, ctx, max_len=W, return_offsets_mapping=True)
        assert np.array_equal(w["offset_mapping"][w["window_off"][:-1]], r["offset_mapping"])
    # a token has the same offsets in every window that holds it
    w = tok.encode_windows(q[:4], ctx[:4], max_len=128, stride=40, return_offsets_mapping=True)
    for d in range(4):
        seen = {}
        for r in range(int(w["window_off"][d]), int(w["window_off"][d + 1])):
            st, n_a = int(w["window_start"][r]), None
            ids = w["input_ids"][r].tolist()
            n_a = ids.index(2) - 1                                        # tokens of the question
            for c in range(n_a + 3, int(w["row_len"][r]) - 1):
                key = st + c - (n_a + 3)
                seen.setdefault(key, tuple(w["offset_mapping"][r, c].tolist()))
                assert seen[key] == tuple(w["offset_mapping"][r, c].tolist())


@gpu
def test_window_offsets_device_form(tok):
    import torch
    from genz_tokenize_b200 import workload
    dev = torch.device("cuda:0")
    up = lambda a: torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)
    from genz_tokenize_b200.tokenizer import pack_strings
    docs = workload.long_documents(workload.default_wordlist().words, 40, lo=50, hi=1500, seed=8)
    q = pack_strings(noisy_rows(41, 40))
    for W, s, paired in ((512, 128, False), (130, 33, True), (98, 0, False)):          # (98: the one-column-per-lane form)
        a, b = (q, docs) if paired else (docs, None)
        host = tok.encode_windows(a, b, max_len=W, stride=s, return_offsets_mapping=True)
        args = [up(a[0]), torch.from_numpy(a[1]).to(dev)] + ([up(b[0]), torch.from_numpy(b[1]).to(dev)] if paired else [None, None])
        got = tok.encode_windows_device(*args, max_len=W, stride=s, text_bytes=len(a[0]), pair_bytes=len(b[0]) if paired else None,
                                        return_offsets_mapping=True)
        torch.cuda.synchronize()
        assert tok.check_errors(dev) == 0
        for k, v in got.items():
            assert np.array_equal(v.cpu().numpy(), host[k]), (W, s, paired, k)
    # a step 2 whose flag differs from step 1's redoes step 1
    lib, st = tok._lib, tok._torch_stream(dev)
    tx, to, nb = up(docs[0]), torch.from_numpy(docs[1]).to(dev), len(docs[0])
    W, s = 64, 8
    n = to.numel() - 1
    wo = torch.empty((n + 1,), dtype=torch.int64, device=dev)
    K = C.c_int64()
    assert lib.genztok_encode_windows_device(tok._h, 0, tx.data_ptr(), to.data_ptr(), nb, None, None, 0, n, W, s, 0, wo.data_ptr(),
                                             None, None, None, C.byref(K), st) == 0
    K = K.value
    ids = torch.empty((K, W), dtype=torch.int32, device=dev); mask = torch.empty((K, W), dtype=torch.uint8, device=dev)
    rl = torch.empty((K,), dtype=torch.int32, device=dev); wd = torch.empty((K,), dtype=torch.int64, device=dev); ws = torch.empty((K,), dtype=torch.int32, device=dev)
    om = torch.full((K, W, 2), -7, dtype=torch.int32, device=dev)
    P = L.DevPlanes(); P.input_ids, P.attention_mask, P.row_len, P.offsets = ids.data_ptr(), mask.data_ptr(), rl.data_ptr(), om.data_ptr()
    assert lib.genztok_encode_windows_device(tok._h, 0, tx.data_ptr(), to.data_ptr(), nb, None, None, 0, n, W, s, L.WANT_OFFSETS, wo.data_ptr(),
                                             C.byref(P), wd.data_ptr(), ws.data_ptr(), None, st) == 0
    torch.cuda.synchronize()
    host = tok.encode_windows(docs, max_len=W, stride=s, return_offsets_mapping=True)
    assert np.array_equal(om.cpu().numpy(), host["offset_mapping"]) and np.array_equal(ids.cpu().numpy(), host["input_ids"])
    # ... and back: a step 2 without the flag after a step 1 with it leaves the offsets plane alone
    om.fill_(-7)
    assert lib.genztok_encode_windows_device(tok._h, 0, tx.data_ptr(), to.data_ptr(), nb, None, None, 0, n, W, s, 0, wo.data_ptr(),
                                             C.byref(P), wd.data_ptr(), ws.data_ptr(), None, st) == 0
    torch.cuda.synchronize()
    assert (om == -7).all() and np.array_equal(ids.cpu().numpy(), host["input_ids"])
    assert tok.check_errors(dev) == 0
