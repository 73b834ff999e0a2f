"""Long documents as overlapping windows (Tokenize.encode_windows / encode_windows_device).

The expected windows are cut here from the oracle's untruncated encodes (one call per side) and put through the reference's
rules on ids: __padding to max_len, the attention mask (ids != pad), and get_sequence_id + get_token_type through
oracle.sequence_id(ids, True) for pairs.  Argument checks and the host-only handle run on the CPU; everything else on the GPU."""
import ctypes as C

import numpy as np
import pytest

from genz_tokenize_b200 import _lib as L

gpu = pytest.mark.gpu


# ---- the expected result, from the oracle -------------------------------------------------------------------------------
def _streams(oracle, side):
    """Every document's token list without its framing: encode(text)[1:-1]."""
    r = oracle.encode_batch(side, None, max_len=None, threads=8)
    ids, off = r["ids"], r["ids_off"]
    return [ids[off[d] + 1:off[d + 1] - 1] for d in range(r["n"])]


def window_count(L_, W, s, LA=None):
    C_ = W - 2 if LA is None else W - LA - 4
    if C_ - s < 1 or L_ <= C_:
        return 1
    return 1 + -(-(L_ - C_) // (C_ - s))


def expected_windows(oracle, texts, pairs, W, s, specials=(0, 1, 2)):
    """dict of the planes encode_windows returns (token types as ids, None as -1) plus the three maps."""
    pad, bos, eos = specials
    A = _streams(oracle, texts)
    B = _streams(oracle, pairs) if pairs is not None else None
    rows, doc, start, off = [], [], [], [0]
    for d in range(len(A)):
        if B is None:
            T, C_ = A[d], W - 2
            K = window_count(len(T), W, s)
            for k in range(K):
                st = k * (C_ - s)
                rows.append([bos] + T[st:st + C_].tolist() + [eos])
                doc.append(d); start.append(st)
        else:
            a, T = A[d].tolist(), B[d]
            C_ = W - len(a) - 4
            K = window_count(len(T), W, s, len(a))
            for k in range(K):
                st = 0 if C_ - s < 1 else k * (C_ - s)
                part = T.tolist() if C_ - s < 1 else T[st:st + C_].tolist()
                rows.append([bos] + a + [eos, eos] + part + [eos])
                doc.append(d); start.append(st)
        off.append(len(rows))
    n = len(rows)
    ids = np.full((n, W), pad, dtype=np.int32)
    row_len = np.zeros(n, dtype=np.int32)
    out = dict(window_off=np.array(off, dtype=np.int64), overflow_to_sample_mapping=np.array(doc, dtype=np.int64),
               window_start=np.array(start, dtype=np.int32))
    for i, r in enumerate(rows):
        if len(r) < W:                                               # __padding (tokenize.py:141-146)
            ids[i, :len(r)] = r
            row_len[i] = len(r)
        else:
            ids[i] = r[:W - 1] + [eos]
            row_len[i] = W
    out.update(input_ids=ids, attention_mask=(ids != pad).astype(np.uint8), row_len=row_len)
    if pairs is not None:
        tt = np.zeros((n, W), dtype=np.int64)
        seq_len = np.zeros(n, dtype=np.int32)
        status = np.zeros(n, dtype=np.uint8)
        for i in range(n):
            try:
                q = [-1 if v is None else v for v in oracle.sequence_id(ids[i], True)]
            except ValueError:
                status[i] = 1
                continue
            seq_len[i] = len(q)
            tt[i] = (q + [pad] * (W - len(q))) if len(q) < W else q[:W - 1] + [eos]
        out.update(token_type_ids=tt, seq_len=seq_len, row_status=status)
    return out


def as_ids(tt8, pad, eos):
    """token_type_ids plane -> ids (the marks of ids that do not fit an int8 -> the ids)."""
    t = np.asarray(tt8).astype(np.int64)
    return np.where(t == L.EOS_MARK, eos, np.where(t == L.PAD_MARK, pad, t))


def assert_windows_equal(got, exp, what, specials=(0, 1, 2)):
    got = {k: (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)) for k, v in got.items()}
    for k in ("window_off", "overflow_to_sample_mapping", "window_start", "input_ids", "attention_mask", "row_len"):
        assert got[k].shape == exp[k].shape, (what, k, got[k].shape, exp[k].shape)
        bad = np.argwhere(got[k] != exp[k])
        assert not len(bad), "%s: %s differs first at %s:\n ours=%s\n ref =%s" % (
            what, k, bad[0], got[k][bad[0][0]].tolist() if got[k].ndim > 1 else got[k][bad[0][0]], exp[k][bad[0][0]].tolist() if exp[k].ndim > 1 else exp[k][bad[0][0]])
    if "row_status" in exp:
        assert np.array_equal(got["row_status"], exp["row_status"]), what
        ok = exp["row_status"] == 0
        assert np.array_equal(got["seq_len"][ok], exp["seq_len"][ok]), what
        tt = as_ids(got["token_type_ids"], specials[0], specials[2])
        bad = np.argwhere((tt != exp["token_type_ids"]) & ok[:, None])
        assert not len(bad), "%s: token_type_ids differ in window %d:\n ours=%s\n ref =%s\n ids =%s" % (
            what, bad[0][0], tt[bad[0][0]].tolist(), exp["token_type_ids"][bad[0][0]].tolist(), got["input_ids"][bad[0][0]].tolist())


# ---- CPU: arguments and the host-only handle -----------------------------------------------------------------------------
def test_window_arguments_rejected():
    from genz_tokenize_b200 import Tokenize
    t = Tokenize(devices=[])
    for W, s in ((2, 0), (0, 0), (16, -1), (16, 14), (16, 20), (3, 1)):
        with pytest.raises(ValueError):
            t.encode_windows(["a b"], max_len=W, stride=s)
    with pytest.raises(ValueError):
        t.encode_windows_device(None, None, max_len=2)
    lib = L.load()
    tb = np.frombuffer(b"a b", dtype=np.uint8).copy()
    to = np.array([0, 3], dtype=np.int64)
    w = L.Windows()
    for W, s in ((2, 0), (16, -1), (16, 14)):
        assert lib.genztok_encode_windows(t._h, tb.ctypes.data, to.ctypes.data, None, None, 1, W, s, 0, C.byref(w)) == L.E_INVALID


def test_windows_host_only_handle_has_no_cpu_path():
    from genz_tokenize_b200 import Tokenize
    from genz_tokenize_b200.tokenizer import GenztokError
    t = Tokenize(devices=[])
    with pytest.raises(GenztokError, match="no CPU path"):
        t.encode_windows(["xin chào"], max_len=16, stride=2)


def test_window_count_formula():
    # K = 1 if L <= C else 1 + ceil((L - C) / (C - s)), C = W - 2
    W, s = 16, 4
    C_ = W - 2
    assert [window_count(L_, W, s) for L_ in (0, C_, C_ + 1, 2 * C_ - s, 2 * C_ - s + 1)] == [1, 1, 2, 2, 3]
    assert window_count(100, 20, 1, LA=15) == 1                     # C_B - s < 1: no room to step, one window
    assert window_count(100, 20, 0, LA=15) == 100
    assert window_count(100, 20, 0, LA=14) == 50


def test_expected_windows_start_with_the_oracle_rows(oracle):
    # the helper's window 0 is the reference's truncated row (the invariant the GPU tests rest on), on the oracle alone
    t, p = _noisy(3, 200, 0, 60), _noisy(4, 200, 0, 60)
    for W, s in ((16, 5), (40, 0)):
        for pairs in (None, p):
            exp = expected_windows(oracle, t, pairs, W, s)
            r = oracle.encode_batch(t, pairs, max_len=W, threads=8)
            first = exp["window_off"][:-1]
            assert np.array_equal(exp["input_ids"][first].reshape(-1), r["ids"])
            assert np.array_equal(exp["attention_mask"][first].reshape(-1), r["mask"])
            if pairs is not None:
                assert np.array_equal(exp["row_status"][first], r["status"])
                ok = r["status"] == 0
                assert np.array_equal(exp["token_type_ids"][first][ok], r["tt"].reshape(-1, W))      # (the oracle lists the rows that do not raise)


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tok():
    from genz_tokenize_b200 import Tokenize
    return Tokenize(devices=[0])


def _noisy(seed, n, lo, hi):
    from genz_tokenize_b200 import workload
    return workload.generate(seed, n, lo, hi, 0.05)


@gpu
@pytest.mark.parametrize("W", [3, 16, 130, 512])
def test_first_window_is_the_truncated_row(tok, W):
    C_ = W - 2
    hi = max(8, W + W // 2)
    for paired in (False, True):
        t = _noisy(900 + W, 300, 0, hi)
        p = _noisy(1900 + W, 300, 0, hi) if paired else None
        ref = tok.encode_batch(t, p, max_len=W, sequence_id=True)
        for s in sorted({0, min(1, C_ - 1), C_ - 1}):
            w = tok.encode_windows(t, p, max_len=W, stride=s, sequence_id=True)
            first = w["window_off"][:-1]
            assert len(w["window_off"]) == 301 and w["window_off"][-1] == len(w["input_ids"])
            assert (np.diff(w["window_off"]) >= 1).all()
            keys = ["input_ids", "attention_mask", "row_len"] + (["token_type_ids", "sequence_id", "seq_len", "row_status"] if paired else [])
            for k in keys:
                assert np.array_equal(w[k][first], ref[k]), (W, s, paired, k)
            assert (w["window_start"][first] == 0).all()


@gpu
def test_windows_match_oracle_short_noisy(tok, oracle):
    for W, s in ((16, 4), (16, 0), (130, 37), (3, 0)):
        t = _noisy(11 + W + s, 600, 0, 3 * W)
        exp = expected_windows(oracle, t, None, W, s)
        assert_windows_equal(tok.encode_windows(t, max_len=W, stride=s), exp, "singles W=%d s=%d" % (W, s))
        p = _noisy(5011 + W + s, 600, 0, 3 * W)
        q = _noisy(7011 + W + s, 600, 0, 6)
        exp = expected_windows(oracle, q, p, W, s)
        assert_windows_equal(tok.encode_windows(q, p, max_len=W, stride=s), exp, "pairs W=%d s=%d" % (W, s))


@gpu
def test_windows_match_oracle_long_documents(tok, oracle):
    from genz_tokenize_b200 import workload
    docs = workload.long_documents(workload.default_wordlist().words, 200)
    exp = expected_windows(oracle, docs, None, 512, 128)
    got = tok.encode_windows(docs, max_len=512, stride=128)
    assert len(got["input_ids"]) > 2000
    assert_windows_equal(got, exp, "200 long documents W=512 s=128")
    # question + long context
    q = _noisy(77, 48, 3, 20)
    ctx = workload.long_documents(workload.default_wordlist().words, 48, lo=300, hi=2500, seed=9)
    exp = expected_windows(oracle, q, ctx, 384, 128)
    got = tok.encode_windows(q, ctx, max_len=384, stride=128)
    assert_windows_equal(got, exp, "QA pairs W=384 s=128")


@gpu
def test_windows_pad_token_is_a_vocab_word(oracle):
    # pad ids that are words (one fits an int8, one does not: PAD_MARK), with literal </s> / <s> / <pad> words in the text so
    # that windows take the k_post_rows row list
    from golden_util import load_padtt_golden
    from genz_tokenize_b200 import Tokenize
    from genz_tokenize_b200.data import bundled_paths
    from oracle.oracle import Oracle
    v, b = bundled_paths()
    rng = np.random.default_rng(4)
    for blk in load_padtt_golden():
        pt = blk["pad_token"]
        t = Tokenize(pad_token=pt, devices=[0])
        o = Oracle(v, b, [pt, None, None, None, None])
        words = ["xin", "chào", "sinh_viên", pt, "</s>", "<s>", "<pad>", "hello", "của", "các"]
        mk = lambda n, lo, hi: [" ".join(rng.choice(words, int(rng.integers(lo, hi)))) for _ in range(n)]
        texts, ctx = mk(300, 0, 60), mk(300, 0, 90)
        sp = (blk["pad_id"], 1, 2)
        for W, s in ((16, 3), (48, 10), (130, 0)):
            assert_windows_equal(t.encode_windows(texts, max_len=W, stride=s), expected_windows(o, texts, None, W, s, sp), "pad %r singles W=%d" % (pt, W), sp)
            assert_windows_equal(t.encode_windows(texts, ctx, max_len=W, stride=s), expected_windows(o, texts, ctx, W, s, sp), "pad %r pairs W=%d" % (pt, W), sp)


@gpu
def test_windows_cover_every_token(tok, oracle):
    from genz_tokenize_b200 import workload
    docs = workload.long_documents(workload.default_wordlist().words, 40, lo=100, hi=900, seed=3)
    T = _streams(oracle, docs)
    for W, s in ((64, 0), (64, 20), (512, 128), (130, 127)):
        w = tok.encode_windows(docs, max_len=W, stride=s)
        off, ids, rl = w["window_off"], w["input_ids"], w["row_len"]
        for d in range(len(T)):
            K = int(off[d + 1] - off[d])
            assert K == window_count(len(T[d]), W, s), (W, s, d)
            rec = []
            for k in range(K):
                r = int(off[d]) + k
                content = ids[r, 1:rl[r] - 1].tolist()
                assert w["window_start"][r] == k * (W - 2 - s)
                rec += content if k == 0 else content[s:]
            assert rec == T[d].tolist(), (W, s, d)


@gpu
def test_windows_edges(tok, oracle):
    W, s = 16, 4
    C_ = W - 2
    one = "sinh_viên"                                                # one token
    assert len(_streams(oracle, [one])[0]) == 1
    docs = ["", "   ", "\n", " \t "] + [" ".join([one] * L_) for L_ in (C_, C_ + 1, 2 * C_ - s, 2 * C_ - s + 1)]
    w = tok.encode_windows(docs, max_len=W, stride=s)
    assert np.diff(w["window_off"]).tolist() == [1, 1, 1, 1, 1, 2, 2, 3]
    for d in range(4):
        assert w.row(int(w["window_off"][d])) == {"input_ids": [1, 2] + [0] * (W - 2), "attention_mask": [1, 1] + [0] * (W - 2)}
    assert_windows_equal(w, expected_windows(oracle, docs, None, W, s), "edges")
    # pairs whose first text leaves no room to step (C_B - s < 1): one window, the encode_batch row, ValueError rows included
    q = [" ".join([one] * k) for k in (7, 8, 9, 10, 11, 12, 13, 20, 40)]
    ctx = [" ".join(["xin chào"] * 30)] * len(q)
    w = tok.encode_windows(q, ctx, max_len=W, stride=s)
    assert (np.diff(w["window_off"])[2:] == 1).all()
    ref = tok.encode_batch(q, ctx, max_len=W)
    first = w["window_off"][:-1]
    for k in ("input_ids", "attention_mask", "token_type_ids", "seq_len", "row_status"):
        assert np.array_equal(w[k][first], ref[k]), k
    assert w["row_status"].any()
    assert_windows_equal(w, expected_windows(oracle, q, ctx, W, s), "pairs without room")


@gpu
def test_windows_device_form_equals_host_form(tok):
    import torch
    from genz_tokenize_b200 import workload
    dev = torch.device("cuda:0")
    up = lambda a: torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)
    docs = workload.long_documents(workload.default_wordlist().words, 64, lo=50, hi=1500, seed=8)
    q = _noisy(31, 64, 0, 30)
    for W, s, paired in ((512, 128, False), (130, 33, True), (96, 0, True)):
        a, b = (q, docs) if paired else (docs, None)
        host = tok.encode_windows(a, b, max_len=W, stride=s, sequence_id=True)
        args = [up(a[0]), torch.from_numpy(a[1]).to(dev)] + ([up(b[0]), torch.from_numpy(b[1]).to(dev)] if paired else [None, None])
        got = tok.encode_windows_device(*args, max_len=W, stride=s, sequence_id=True, text_bytes=len(a[0]), pair_bytes=len(b[0]) if paired else None)
        torch.cuda.synchronize()
        assert tok.check_errors(dev) == 0
        for k, v in got.items():
            assert np.array_equal(v.cpu().numpy(), host[k]), (W, s, paired, k)
    # step 2 after a step 1 for another batch redoes step 1
    lib = tok._lib
    st = tok._torch_stream(dev)
    bat = [(up(x[0]), torch.from_numpy(x[1]).to(dev), len(x[0])) for x in (docs, _noisy(32, 200, 0, 900))]
    W, s = 64, 8
    offs, Ks = [], []
    for tx, to, nb in bat:
        wo = torch.empty((to.numel(),), dtype=torch.int64, device=dev)
        K = C.c_int64()
        assert lib.genztok_encode_windows_device(tok._h, 0, tx.data_ptr(), to.data_ptr(), nb, None, None, 0, to.numel() - 1, W, s, 0, wo.data_ptr(),
                                                 None, None, None, C.byref(K), st) == 0
        offs.append(wo); Ks.append(K.value)
    tx, to, nb = bat[0]
    K = Ks[0]
    ids = torch.empty((K, W), dtype=torch.int32, device=dev); mask = torch.empty((K, W), dtype=torch.uint8, device=dev)
    rl = torch.empty((K,), dtype=torch.int32, device=dev); wd = torch.empty((K,), dtype=torch.int64, device=dev); ws = torch.empty((K,), dtype=torch.int32, device=dev)
    P = L.DevPlanes(); P.input_ids, P.attention_mask, P.row_len = ids.data_ptr(), mask.data_ptr(), rl.data_ptr()
    assert lib.genztok_encode_windows_device(tok._h, 0, tx.data_ptr(), to.data_ptr(), nb, None, None, 0, to.numel() - 1, W, s, 0, offs[0].data_ptr(),
                                             C.byref(P), wd.data_ptr(), ws.data_ptr(), None, st) == 0
    torch.cuda.synchronize()
    host = tok.encode_windows(docs, max_len=W, stride=s)
    assert np.array_equal(ids.cpu().numpy(), host["input_ids"]) and np.array_equal(mask.cpu().numpy(), host["attention_mask"])
    assert np.array_equal(wd.cpu().numpy(), host["overflow_to_sample_mapping"]) and np.array_equal(offs[0].cpu().numpy(), host["window_off"])
    assert tok.check_errors(dev) == 0


@gpu
def test_windows_chunking_sharding_and_launches(oracle):
    import torch
    from genz_tokenize_b200 import DataCollection, Tokenize, workload
    docs = workload.long_documents(workload.default_wordlist().words, 50, lo=20, hi=1200, seed=6)
    q = _noisy(41, 50, 0, 25)
    base = Tokenize(devices=[0])
    small = Tokenize(devices=[0])
    small.set_option("chunk_rows", 7)
    for a, b in ((docs, None), (q, docs)):
        x, y = base.encode_windows(a, b, max_len=128, stride=32), small.encode_windows(a, b, max_len=128, stride=32)
        assert set(x) == set(y)
        for k in x:
            assert np.array_equal(np.asarray(x[k]), np.asarray(y[k])), k
    # kernel launches per call: fixed for a chunk, whatever its number of documents
    counts = []
    for n in (10, 1000):
        t = _noisy(51, n, 0, 300)
        c0 = base.launch_count()
        base.encode_windows(t, max_len=64, stride=16)
        counts.append(base.launch_count() - c0)
    assert counts[0] == counts[1], counts
    # hand-off: one label per window
    w = base.encode_windows(q, docs, max_len=128, stride=32)
    labels = np.arange(50)
    dc = DataCollection.from_encoding(w, y=labels[w["overflow_to_sample_mapping"]])
    assert len(dc) == len(w["input_ids"])
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    multi = Tokenize(devices=list(range(ndev)))
    for a, b in ((docs, None), (q, docs)):
        x, y = base.encode_windows(a, b, max_len=128, stride=32), multi.encode_windows(a, b, max_len=128, stride=32)
        for k in x:
            assert np.array_equal(np.asarray(x[k]), np.asarray(y[k])), k
