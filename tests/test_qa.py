"""Extractive QA over the windows' planes: Tokenize.qa_labels and Tokenize.qa_best_spans.

The expected values come from a numpy restatement of the semantics (include/genztok.h) below, which follows the definitions
literally: context columns from the offsets alone, labels from the overlapping context columns, best spans by a search over every
(window, s, e).  The windows' offsets and window_off come from the library, which tests/test_offsets.py pins against the oracle.
The restatement and the argument checks run on the CPU; everything else on the GPU."""
import re

import numpy as np
import pytest

from genz_tokenize_b200 import _lib as L

gpu = pytest.mark.gpu
WORD = re.compile(r"\S+\n?")


# ---- the restatement ----------------------------------------------------------------------------------------------------------
def context_cols(row, pair):
    """Context columns of one window [W, 2]: singles, end > 0; pairs, end > 0 after z, the first column >= 1 that is (0, 0)."""
    W = len(row)
    if pair:
        z = next((c for c in range(1, W) if row[c, 0] == 0 and row[c, 1] == 0), None)
        if z is None:
            return []
        return [c for c in range(z + 1, W) if row[c, 1] > 0]
    return [c for c in range(W) if row[c, 1] > 0]


def ref_labels(om, win_off, pair, answers):
    K = len(om)
    st, en = np.zeros(K, dtype=np.int64), np.zeros(K, dtype=np.int64)
    for d in range(len(win_off) - 1):
        a0, a1 = int(answers[d][0]), int(answers[d][1])
        for i in range(int(win_off[d]), int(win_off[d + 1])):
            if a1 <= a0:
                continue
            cols = [c for c in context_cols(om[i], pair) if om[i, c, 0] < a1 and om[i, c, 1] > a0]
            if cols and om[i, cols[0], 0] <= a0 and om[i, cols[-1], 1] >= a1:
                st[i], en[i] = cols[0], cols[-1]
    return st, en


def ref_spans(S, E, om, win_off, pair, L_):
    n = len(win_off) - 1
    out = {"score": np.full(n, -np.inf, dtype=np.float32), "null_score": np.full(n, np.nan, dtype=np.float32),
           "window": np.full(n, -1, dtype=np.int64), "columns": np.zeros((n, 2), dtype=np.int32), "span": np.zeros((n, 2), dtype=np.int32)}
    for d in range(n):
        best = None
        for i in range(int(win_off[d]), int(win_off[d + 1])):
            out["null_score"][d] = np.fmin(out["null_score"][d], np.float32(S[i, 0]) + np.float32(E[i, 0]))
            ctx = context_cols(om[i], pair)
            if not ctx:
                continue
            cols = np.array(ctx)
            sc = S[i, cols][:, None].astype(np.float32) + E[i, cols][None, :].astype(np.float32)
            s_, e_ = np.meshgrid(cols, cols, indexing="ij")
            ok = (e_ >= s_) & (e_ - s_ + 1 <= L_) & ~np.isnan(sc)
            if not ok.any():
                continue
            m = sc[ok].max()
            a, b = np.argwhere(ok & (sc == m))[0]                      # row-major: the smallest s, then e
            if best is None or m > best[0]:
                best = (m, i, int(cols[a]), int(cols[b]))
        if best is not None:
            m, i, s, e = best
            out["score"][d], out["window"][d], out["columns"][d] = m, i, (s, e)
            out["span"][d] = (om[i, s, 0], om[i, e, 1])
    return out


def char_to_byte(t, k):
    """unit='char' on the host: Python str index -> byte position ('surrogatepass' UTF-8)."""
    cb = np.concatenate([[0], np.cumsum([len(ch.encode("utf-8", "surrogatepass")) for ch in t])]).astype(np.int64)
    if k < 0:
        return k
    return int(cb[k]) if k <= len(t) else int(cb[-1]) + (k - len(t))


def make_answers(rng, texts):
    """Byte spans of every kind: word-aligned runs, spans that start or end mid-token or in whitespace, empty and reversed spans,
    spans past the end, the whole text."""
    out = []
    for t in texts:
        b = t.encode("utf-8", "surrogatepass")
        n = len(b)
        cb = np.concatenate([[0], np.cumsum([len(ch.encode("utf-8", "surrogatepass")) for ch in t])]).astype(np.int64)
        words = [(int(cb[m.start()]), int(cb[m.start() + len(m.group(0).rstrip(chr(10)))])) for m in WORD.finditer(t)]
        kind = int(rng.integers(0, 8))
        if kind <= 2 and words:
            i = int(rng.integers(0, len(words)))
            j = min(len(words) - 1, i + int(rng.integers(0, 6)))
            a = (words[i][0], words[j][1])
        elif kind == 3 and n:
            a0 = int(rng.integers(0, n))
            a = (a0, a0 + int(rng.integers(1, 40)))
        elif kind == 4:
            a0 = int(rng.integers(0, n + 1))
            a = (a0, a0 - int(rng.integers(0, 3)))
        elif kind == 5:
            a = (n + int(rng.integers(0, 3)), n + 10)
        elif kind == 6:
            a = (0, n)
        else:
            a0 = int(rng.integers(0, n + 1))
            a = (a0, min(n, a0 + int(rng.integers(1, 200))))
        out.append(a)
    return np.array(out, dtype=np.int64).reshape(-1, 2)


# ---- CPU: the restatement on hand-worked windows --------------------------------------------------------------------------------
Z = (0, 0)


def rows(*r, W=None):
    W = W or max(len(x) for x in r)
    return np.array([list(x) + [Z] * (W - len(x)) for x in r], dtype=np.int32)


def test_restatement_readme_vector():
    # tok("sinh_viên công_nghệ", "hello", max_len=10): [<s>] A [</s> </s>] B [</s>] pads
    om = rows([Z, (0, 10), (11, 23), Z, Z, (0, 5), Z, Z, Z, Z])
    assert context_cols(om[0], True) == [5]
    assert context_cols(om[0], False) == [1, 2, 5]
    wo = np.array([0, 1])
    assert [x.tolist() for x in ref_labels(om, wo, True, [(0, 5)])] == [[5], [5]]
    assert [x.tolist() for x in ref_labels(om, wo, True, [(1, 3)])] == [[5], [5]]        # inside the token
    assert [x.tolist() for x in ref_labels(om, wo, True, [(0, 6)])] == [[0], [0]]        # past the end
    assert [x.tolist() for x in ref_labels(om, wo, True, [(3, 3)])] == [[0], [0]]        # no answer
    assert [x.tolist() for x in ref_labels(rows(om[0]), wo, False, [(11, 23)])] == [[2], [2]]
    S = np.zeros((1, 10), dtype=np.float32)
    E = np.zeros((1, 10), dtype=np.float32)
    r = ref_spans(S, E, om, wo, True, 30)
    assert r["window"].tolist() == [0] and r["columns"].tolist() == [[5, 5]] and r["span"].tolist() == [[0, 5]] and r["null_score"][0] == 0


def test_restatement_pair_empty_question_and_full_row():
    # an empty question: [<s>] [</s> </s>] B [</s>]
    om = rows([Z, Z, Z, (0, 3), (4, 9), Z, Z, Z])
    assert context_cols(om[0], True) == [3, 4]
    # a question that fills the row: no context, no label, no candidate
    full = rows([Z, (0, 2), (3, 5), (6, 8), (9, 11), (12, 14), (15, 17), Z])
    assert context_cols(full[0], True) == []
    assert [x.tolist() for x in ref_labels(full, np.array([0, 1]), True, [(0, 2)])] == [[0], [0]]
    r = ref_spans(np.ones((1, 8), np.float32), np.ones((1, 8), np.float32), full, np.array([0, 1]), True, 30)
    assert r["window"].tolist() == [-1] and r["score"][0] == -np.inf and r["null_score"][0] == 2


def test_restatement_stride_overlap():
    # two windows of one single with stride 1: tokens (0,2) (3,5) (6,8) | (6,8) (9,11)
    om = rows([Z, (0, 2), (3, 5), (6, 8), Z], [Z, (6, 8), (9, 11), Z, Z])
    wo = np.array([0, 2])
    st, en = ref_labels(om, wo, False, [(6, 8)])                       # in the overlap: labelled in both windows
    assert st.tolist() == [3, 1] and en.tolist() == [3, 1]
    st, en = ref_labels(om, wo, False, [(3, 11)])                      # crosses the border: in neither
    assert st.tolist() == [0, 0] and en.tolist() == [0, 0]
    S = np.array([[0, 0, 0, 5, 0], [0, 5, 0, 0, 0]], np.float32)
    E = np.array([[0, 0, 0, 5, 0], [0, 5, 0, 0, 0]], np.float32)
    r = ref_spans(S, E, om, wo, False, 30)
    assert r["window"].tolist() == [0] and r["columns"].tolist() == [[3, 3]]   # the tie goes to the smaller window


def test_char_to_byte_restatement():
    t = "đi \U0001F600x\ud800y"
    assert [char_to_byte(t, k) for k in range(len(t) + 3)] == [0, 2, 3, 4, 8, 9, 12, 13, 14, 15]
    assert char_to_byte(t, -2) == -2


# ---- CPU: argument checks through the C ABI and the host-only handle ----------------------------------------------------------
def test_qa_argument_checks_and_host_only_handle():
    from genz_tokenize_b200 import Tokenize
    from genz_tokenize_b200.tokenizer import GenztokError
    t = Tokenize(devices=[])
    lib = L.load()
    buf = np.zeros(4096, dtype=np.uint8)
    p = buf.ctypes.data                                                # stands for device pointers: nothing is launched
    lab = lambda **kw: lib.genztok_qa_labels_device(t._h, 0, kw.get("om", p), 4, kw.get("W", 16), 0, kw.get("wo", p), 2, kw.get("ans", p),
                                                    kw.get("unit", L.QA_BYTES), kw.get("text", None), kw.get("toff", None), 0,
                                                    kw.get("st", p), p, None)
    assert lab(W=2) == L.E_INVALID
    assert lab(unit=7) == L.E_INVALID
    assert lab(unit=L.QA_CHARS) == L.E_INVALID                          # characters need the text
    assert lab(st=None) == L.E_INVALID
    assert lab(wo=None) == L.E_INVALID
    assert lab() == L.E_NODEVICE
    assert lab(unit=L.QA_CHARS, text=p, toff=p) == L.E_NODEVICE
    spans = lambda **kw: lib.genztok_qa_best_spans_device(t._h, 0, p, p, p, 4, kw.get("W", 16), 1, p, 2, kw.get("L", 30), kw.get("score", p), p, p, p, p, None)
    assert spans(W=2) == L.E_INVALID
    assert spans(L=0) == L.E_INVALID
    assert spans(score=None) == L.E_INVALID
    assert spans() == L.E_NODEVICE
    assert b"no such device" in lib.genztok_last_error(t._h)
    enc = {"offset_mapping": np.zeros((2, 8, 2), np.int32), "window_off": np.array([0, 2])}
    with pytest.raises(GenztokError, match="no CPU path"):
        t.qa_labels(enc, np.zeros((1, 2), np.int64))
    with pytest.raises(ValueError, match="offset_mapping"):
        t.qa_labels({"input_ids": np.zeros((2, 8), np.int32)}, np.zeros((2, 2), np.int64))
    with pytest.raises(ValueError, match="ragged"):
        t.qa_labels({"offset_mapping": np.zeros((9, 2), np.int32)}, np.zeros((2, 2), np.int64))
    with pytest.raises(ValueError, match="unit"):
        t.qa_labels(enc, np.zeros((1, 2), np.int64), unit="word")
    with pytest.raises(ValueError, match="max_answer_len"):
        t.qa_best_spans(enc, np.zeros((2, 8)), np.zeros((2, 8)), max_answer_len=0)


# ---- GPU --------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tok():
    from genz_tokenize_b200 import Tokenize
    return Tokenize(devices=[0])


def singles(W):
    from test_offsets import noisy_rows
    return noisy_rows(100 + W, 160)


def qa_pairs(n, seed):
    """Questions (some with a literal </s>, some empty, some long enough to fill small windows) + long noisy contexts."""
    from genz_tokenize_b200 import workload
    from test_offsets import WS, noisy_rows, unpack
    q = noisy_rows(seed, n)
    q = [("</s> " + x if i % 5 == 0 else x + " </s> đâu" if i % 5 == 1 else x) for i, x in enumerate(q)]
    q[2] = ""
    ctx = unpack(workload.long_documents(workload.default_wordlist().words, n, lo=40, hi=600, seed=seed))
    ctx = [c + WS[i % 29] + noisy_rows(seed + 1 + i, 1)[0] for i, c in enumerate(ctx)]
    return q, ctx


def check_labels(tok, w, texts, answers, pair, what):
    om, wo = w["offset_mapping"], w["window_off"]
    st, en = tok.qa_labels(w, answers)
    es, ee = ref_labels(om, wo, pair, answers)
    bad = np.flatnonzero((st != es) | (en != ee))
    assert not len(bad), "%s: window %d: ours (%d, %d), ref (%d, %d)" % (what, bad[0], st[bad[0]], en[bad[0]], es[bad[0]], ee[bad[0]])
    # round trip: the labelled columns' bytes hold the answer
    doc = w["overflow_to_sample_mapping"]
    for i in np.flatnonzero(st):
        d = int(doc[i])
        a0, a1 = answers[d]
        x, y = om[i, st[i], 0], om[i, en[i], 1]
        assert x <= a0 and y >= a1, (what, i)
        b = texts[d].encode("utf-8", "surrogatepass")
        assert b[a0:a1] in b[x:y]
    return st, en


@gpu
@pytest.mark.parametrize("W", [16, 130, 384, 512])
def test_labels_singles(tok, W):
    texts = singles(W)
    rng = np.random.default_rng(W)
    for s in (0, max(1, (W - 2) // 3)):
        w = tok.encode_windows(texts, max_len=W, stride=s, return_offsets_mapping=True)
        st, _ = check_labels(tok, w, texts, make_answers(rng, texts), False, "singles W=%d s=%d" % (W, s))
        assert tok.check_errors() == 0
        assert st.dtype == np.int64 and st.shape == (len(w["input_ids"]),)


@gpu
@pytest.mark.parametrize("W", [16, 130, 384, 512])
def test_labels_pairs(tok, W):
    q, ctx = qa_pairs(40, 50 + W)
    rng = np.random.default_rng(W + 1)
    for s in (0, max(1, W // 4)):
        if s >= W - 2:
            continue
        w = tok.encode_windows(q, ctx, max_len=W, stride=s, return_offsets_mapping=True)
        answers = make_answers(rng, ctx)
        st, _ = check_labels(tok, w, ctx, answers, True, "pairs W=%d s=%d" % (W, s))
        assert tok.check_errors() == 0
        if W >= 130:
            assert st.any()
    # a question with a literal </s> moves the token types; the context rule does not follow them
    w = tok.encode_windows(["hỏi </s> gì"], ["sinh_viên công_nghệ"], max_len=W, return_offsets_mapping=True)
    st, en = tok.qa_labels(w, np.array([[11, 23]]))
    assert int(st[0]) > 0 and [x.tolist() for x in (st, en)] == [x.tolist() for x in ref_labels(w["offset_mapping"], w["window_off"], True, [(11, 23)])]


@gpu
def test_labels_chars_equal_host_conversion(tok):
    import torch
    from genz_tokenize_b200.tokenizer import pack_strings
    q, ctx = qa_pairs(60, 7)
    rng = np.random.default_rng(3)
    w = tok.encode_windows(q, ctx, max_len=130, stride=40, return_offsets_mapping=True)
    ch = []
    for t in ctx:
        k0 = int(rng.integers(-1, len(t) + 3))
        ch.append((k0, k0 + int(rng.integers(-1, 60))))
    ch[0] = (0, len(ctx[0]))
    ch[1] = (len(ctx[1]), len(ctx[1]) + 2)
    ch = np.array(ch, dtype=np.int64)
    by = np.array([(char_to_byte(t, a), char_to_byte(t, b)) for t, (a, b) in zip(ctx, ch)], dtype=np.int64)
    exp = tok.qa_labels(w, by)
    for context in (ctx, pack_strings(ctx)):
        got = tok.qa_labels(w, ch, unit="char", context=context)
        assert np.array_equal(got[0], exp[0]) and np.array_equal(got[1], exp[1])
    # device form: the text as CUDA tensors
    dev = torch.device("cuda:0")
    b, o = pack_strings(ctx)
    tx = torch.from_numpy(np.concatenate([b, np.zeros((-len(b)) % 16 + 32, dtype=np.uint8)])).to(dev)
    dw = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in w.items() if isinstance(v, np.ndarray)}
    got = tok.qa_labels(dw, torch.from_numpy(ch).to(dev), unit="char", context=(tx, torch.from_numpy(o).to(dev)))
    assert np.array_equal(got[0].cpu().numpy(), exp[0]) and np.array_equal(got[1].cpu().numpy(), exp[1])
    assert tok.check_errors(dev) == 0


@gpu
def test_host_form_equals_device_form(tok):
    import torch
    from genz_tokenize_b200.tokenizer import pack_strings
    dev = torch.device("cuda:0")
    up = lambda a: torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)
    q, ctx = qa_pairs(30, 11)
    a, b = pack_strings(q), pack_strings(ctx)
    W, s = 384, 128
    host = tok.encode_windows(a, b, max_len=W, stride=s, return_offsets_mapping=True)
    out = tok.encode_windows_device(up(a[0]), torch.from_numpy(a[1]).to(dev), up(b[0]), torch.from_numpy(b[1]).to(dev), max_len=W, stride=s,
                                    text_bytes=len(a[0]), pair_bytes=len(b[0]), return_offsets_mapping=True)
    answers = make_answers(np.random.default_rng(5), ctx)
    hs, he = tok.qa_labels(host, answers)
    ds, de = tok.qa_labels(out, torch.from_numpy(answers).to(dev))
    assert ds.device == dev and np.array_equal(ds.cpu().numpy(), hs) and np.array_equal(de.cpu().numpy(), he)
    g = torch.Generator().manual_seed(1)
    S, E = torch.randn(host["input_ids"].shape, generator=g), torch.randn(host["input_ids"].shape, generator=g)
    db = tok.qa_best_spans(out, S.to(dev).double(), E.to(dev).half().float())                       # .float() of other dtypes
    E16 = E.half().float().numpy()
    hb16 = tok.qa_best_spans(host, S.numpy(), E16)
    for k in hb16:
        assert np.array_equal(db[k].cpu().numpy(), hb16[k], equal_nan=True), k
    # encode_batch with offsets: one window per document, equal to window 0 of its windows
    r = tok.encode_batch(q, ctx, max_len=W, return_offsets_mapping=True)
    bs, be = tok.qa_labels(r, answers)
    w0 = host["window_off"][:-1]
    assert np.array_equal(bs, hs[w0]) and np.array_equal(be, he[w0])
    rb = tok.qa_best_spans(r, S.numpy()[w0], E.numpy()[w0])
    exp = ref_spans(S.numpy()[w0], E.numpy()[w0], r["offset_mapping"], np.arange(len(q) + 1), True, 30)
    for k in exp:
        assert np.array_equal(rb[k], exp[k], equal_nan=True), k
    assert tok.check_errors(dev) == 0


def assert_spans(got, exp, what):
    for k in exp:
        g, e = np.asarray(got[k]), exp[k]
        assert g.dtype == e.dtype and np.array_equal(g, e, equal_nan=True), "%s %s:\n ours=%s\n ref =%s" % (what, k, g[:8].tolist(), e[:8].tolist())


@gpu
@pytest.mark.parametrize("W", [16, 130, 384])
def test_best_spans_equal_brute_force(tok, W):
    q, ctx = qa_pairs(40, 90 + W)
    texts = singles(W)[:60]
    rng = np.random.default_rng(W)
    for w, pair in ((tok.encode_windows(q, ctx, max_len=W, stride=min(W // 4, W - 3), return_offsets_mapping=True), True),
                    (tok.encode_windows(texts, max_len=W, stride=W // 3, return_offsets_mapping=True), False)):
        K = len(w["input_ids"])
        for L_ in (1, 3, 30, W):
            S = rng.integers(-3, 4, size=(K, W)).astype(np.float32)           # integer logits: ties everywhere
            E = rng.integers(-3, 4, size=(K, W)).astype(np.float32)
            got = tok.qa_best_spans(w, S, E, max_answer_len=L_)
            assert_spans(got, ref_spans(S, E, w["offset_mapping"], w["window_off"], pair, L_), "W=%d pair=%s L=%d" % (W, pair, L_))
        # -inf and NaN logits, a document whose every window is -inf, random floats
        S = rng.standard_normal((K, W)).astype(np.float32)
        E = rng.standard_normal((K, W)).astype(np.float32)
        S[rng.random((K, W)) < 0.2] = -np.inf
        E[rng.random((K, W)) < 0.2] = -np.inf
        S[rng.random((K, W)) < 0.05] = np.nan
        E[rng.random((K, W)) < 0.05] = np.inf
        S[w["window_off"][1]:w["window_off"][2]] = -np.inf
        E[w["window_off"][3]:w["window_off"][4]] = np.nan
        got = tok.qa_best_spans(w, S, E, max_answer_len=7)
        assert_spans(got, ref_spans(S, E, w["offset_mapping"], w["window_off"], pair, 7), "W=%d pair=%s special values" % (W, pair))
    assert tok.check_errors() == 0


@gpu
def test_best_spans_no_candidate(tok):
    # questions that fill the row: no context in any window
    q = ["từ " * 40] * 3
    w = tok.encode_windows(q, ["sinh_viên công_nghệ"] * 3, max_len=16, return_offsets_mapping=True)
    S = np.ones((len(w["input_ids"]), 16), np.float32)
    got = tok.qa_best_spans(w, S, S)
    assert got["window"].tolist() == [-1] * 3 and np.all(got["score"] == -np.inf) and not got["span"].any() and not got["columns"].any()
    assert np.all(got["null_score"] == 2)
    assert tok.check_errors() == 0


@gpu
def test_labels_to_logits_to_spans(tok):
    q, ctx = qa_pairs(50, 21)
    w = tok.encode_windows(q, ctx, max_len=130, stride=60, return_offsets_mapping=True)
    answers = make_answers(np.random.default_rng(9), ctx)
    st, en = tok.qa_labels(w, answers)
    K, W = w["input_ids"].shape
    S = np.zeros((K, W), np.float32)
    E = np.zeros((K, W), np.float32)
    S[np.arange(K), st] = 10
    E[np.arange(K), en] = 10
    got = tok.qa_best_spans(w, S, E, max_answer_len=W)
    wo = w["window_off"]
    for d in range(len(ctx)):
        lab = [i for i in range(wo[d], wo[d + 1]) if st[i] > 0]
        if not lab:
            continue
        i = lab[0]                                                     # the tie between windows goes to the first
        assert got["window"][d] == i and tuple(got["columns"][d]) == (st[i], en[i]) and got["score"][d] == 20
        a0, a1 = answers[d]
        x, y = got["span"][d]
        assert x <= a0 and y >= a1 and (x, y) == (w["offset_mapping"][i, st[i], 0], w["offset_mapping"][i, en[i], 1])
    assert tok.check_errors() == 0


@gpu
def test_launches_and_errors(tok):
    import torch
    dev = torch.device("cuda:0")
    q, ctx = qa_pairs(20, 31)
    w = tok.encode_windows(q, ctx, max_len=64, stride=8, return_offsets_mapping=True)
    dw = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in w.items() if isinstance(v, np.ndarray)}
    ans = torch.from_numpy(make_answers(np.random.default_rng(1), ctx)).to(dev)
    n0 = tok.launch_count()
    tok.qa_labels(dw, ans)
    assert tok.launch_count() - n0 <= 1
    from genz_tokenize_b200.tokenizer import pack_strings
    b, o = pack_strings(ctx)
    n0 = tok.launch_count()
    tok.qa_labels(w, np.zeros((len(ctx), 2), np.int64), unit="char", context=(b, o))
    assert tok.launch_count() - n0 <= 2
    S = torch.randn(dw["input_ids"].shape, device=dev)
    n0 = tok.launch_count()
    r1 = tok.qa_best_spans(dw, S, S)
    assert tok.launch_count() - n0 <= 2
    r2 = tok.qa_best_spans(dw, S, S)
    for k in r1:
        assert torch.equal(r1[k], r2[k]), k                            # bit-identical from run to run
    assert tok.check_errors(dev) == 0
    # offsets that break the layout are counted, never a fault
    from genz_tokenize_b200 import Tokenize
    t = Tokenize(devices=[0])
    bad = dict(dw)
    bad["offset_mapping"] = dw["offset_mapping"].clone()
    bad["offset_mapping"][0, 0] = 5
    t.qa_labels(bad, ans)
    from genz_tokenize_b200.tokenizer import GenztokError
    with pytest.raises(GenztokError, match="inconsistencies"):
        t.check_errors(dev)


@gpu
def test_integration_snippet_runs():
    # the QA snippet of INTEGRATION.md, as written, against the bundled vocab
    import os
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "INTEGRATION.md"), encoding="utf-8").read()
    block = text[text.index("Extractive QA on the GPU"):]
    block = block[block.index("```python") + len("```python"):]
    block = block[:block.index("```")]
    env = {}
    exec(compile(block, "INTEGRATION.md", "exec"), env)
    w, st, en = env["w"], int(env["start_positions"][0]), int(env["end_positions"][0])
    assert st > 0 and w["offset_mapping"][0, st, 0] == 0 and w["offset_mapping"][0, en, 1] == 3
    assert env["best"]["window"][0] == 0 and 0 <= env["a0"] < env["a1"] <= len(env["contexts"][0].encode())
