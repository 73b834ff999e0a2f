"""BPE-dropout for fixed-layout encodes: encode_batch / encode_device(..., bpe_dropout=p, seed, row_keys) and bpe(..., dropout=p).

The expected rows come from a pure-Python restatement of the rule include/genztok.h states: the \\S+\\n? words of the
'surrogatepass' text, subword-nmt's merge loop with the hash draws, pieces to ids through encoder.get with unk, then the
reference's row (cut, padded, token types through oracle.sequence_id).  Hand-worked words pin the merge loop, and at p = 0 it
equals the oracle's bpe() over the vocab's words.  The restatement and the argument checks run on the CPU; everything else on the GPU."""
import ctypes as C
import math
import re

import numpy as np
import pytest

from genz_tokenize_b200 import _lib as L

gpu = pytest.mark.gpu
GOLD, KEY = 0x9E3779B97F4A7C15, 0x6270655F64726F70
M64 = 2 ** 64 - 1


# ---- the restatement ------------------------------------------------------------------------------------------------------
def mix(x):
    x ^= x >> 30; x = (x * 0xBF58476D1CE4E5B9) & M64; x ^= x >> 27; x = (x * 0x94D049BB133111EB) & M64; x ^= x >> 31
    return x


def thr_of(p):
    return math.floor(p * 2 ** 32)


def word_key(seed, key, j, side):
    """W_j of include/genztok.h."""
    R = mix((mix((seed & M64) ^ KEY) + (key & M64) * GOLD) & M64)
    return mix((R + (2 * j + side + 1) * GOLD) & M64)


def hash_drop(Wj, thr):
    return lambda t, i: (mix((Wj + ((t << 32) | i)) & M64) >> 32) < thr


def merge(word, ranks, dropped):
    """subword-nmt's encode() with dropout: the final symbols of `word` (a str), "</w>" on the last."""
    syms = list(word[:-1]) + [word[-1] + "</w>"]
    t = 0
    while len(syms) > 1:
        pairs = [(ranks[(syms[i], syms[i + 1])], i) for i in range(len(syms) - 1) if (syms[i], syms[i + 1]) in ranks and not dropped(t, i)]
        if not pairs:
            break
        best = min(pairs)[0]
        out, i = [], 0
        for _, j in sorted(p for p in pairs if p[0] == best):
            if j < i:                                               # overlaps the occurrence merged before it (x x x -> xx x)
                continue
            out.extend(syms[i:j])
            out.append(syms[j] + syms[j + 1])
            i = j + 2
        out.extend(syms[i:])
        syms = out
        t += 1
    return syms


class Rule:
    def __init__(self, tok):
        self.ranks, self.enc = tok.bpe_ranks, tok.encoder
        self.pad, self.bos, self.eos, _, self.unk = tok._special_ids()

    def ids(self, syms):
        return [self.enc.get(s + "@@", self.unk) for s in syms[:-1]] + [self.enc.get(syms[-1][:-4], self.unk)]

    def text_ids(self, text, p, seed, key, side, cap):
        """The first `cap` ids of `text` (bytes or str) under dropout."""
        if isinstance(text, bytes):
            text = text.decode("utf-8", "surrogatepass")
        out, thr = [], thr_of(p)
        for j, w in enumerate(re.findall(r"\S+\n?", text)):
            if len(out) >= cap:
                break
            out += self.ids(merge(w, self.ranks, hash_drop(word_key(seed, key, j, side), thr)))
        return out[:cap]

    def rows(self, oracle, texts, pairs, W, p, seed, keys=None):
        """The planes encode_batch(..., bpe_dropout=p) returns (token types as ids, None as -1)."""
        n = len(texts)
        keys = list(range(n)) if keys is None else [int(k) for k in keys]
        ids = np.full((n, W), self.pad, dtype=np.int32)
        row_len = np.zeros(n, dtype=np.int32)
        status = np.zeros(n, dtype=np.uint8)
        tt = np.zeros((n, W), dtype=np.int64)
        seq = np.full((n, W), -2, dtype=np.int64)
        seq_len = np.zeros(n, dtype=np.int32)
        for d in range(n):
            a = self.text_ids(texts[d], p, seed, keys[d], 0, W)
            r = [self.bos] + a + [self.eos]
            if pairs is not None:
                r += [self.eos] + self.text_ids(pairs[d], p, seed, keys[d], 1, W) + [self.eos]
            r = r if len(r) <= W else r[:W - 1] + [self.eos]           # __padding (tokenize.py:141-146)
            ids[d, :len(r)] = r
            row_len[d] = len(r)
            if pairs is None:
                continue
            try:
                q = [-1 if v is None else v for v in oracle.sequence_id(ids[d], True)]
            except ValueError:
                status[d] = 1
            else:
                seq_len[d] = len(q)
                seq[d, :len(q)] = q
                tt[d] = (q + [self.pad] * (W - len(q))) if len(q) < W else q[:W - 1] + [self.eos]
        out = dict(input_ids=ids, attention_mask=(ids != self.pad).astype(np.uint8), row_len=row_len)
        if pairs is not None:
            out.update(token_type_ids=tt, sequence_id=seq, seq_len=seq_len, row_status=status)
        return out


def strs(packed):
    b, o = packed
    return [bytes(b[o[i]:o[i + 1]]).decode("utf-8", "surrogatepass") for i in range(len(o) - 1)]


# ---- CPU: the restatement, the oracle, arguments ------------------------------------------------------------------------
XR = {("x", "x"): 0, ("x", "x</w>"): 1, ("xx", "xx"): 2, ("xx", "xx</w>"): 3}


def test_merge_loop_hand_worked_words():
    never = lambda t, i: False
    drop = lambda *ti: (lambda t, i: (t, i) in ti)
    # x x x x</w>: greedy from the left, a run of equal pairs merges every second occurrence
    assert merge("xxxx", XR, never) == ["xxxx</w>"]                   # [xx x x</w>] -> [xx xx</w>] -> [xxxx</w>]
    assert merge("xxxx", XR, drop((0, 0))) == ["x", "xx", "x</w>"]    # only (x, x) at 1 merges; then nothing has a rank
    assert merge("xxxx", XR, drop((0, 1))) == ["xxxx</w>"]            # the dropped middle occurrence is the one greedy skips
    # x x x x x</w>: a dropped middle occurrence splits the run; both neighbours merge
    assert merge("xxxxx", XR, drop((0, 1))) == merge("xxxxx", XR, never) == ["xxxx", "x</w>"]
    assert merge("xxxxx", XR, drop((0, 0))) == ["x", "xxxx</w>"]     # [x xx x x</w>] -> [x xx xx</w>] -> [x xxxx</w>]
    assert merge("xxxxx", XR, drop((0, 0), (1, 2))) == ["x", "xx", "x", "x</w>"]   # round 1 drops its only candidate: final
    # a round where every pair is dropped ends the word (no retry); a one-code-point word has no pair
    assert merge("xxxx", XR, lambda t, i: True) == ["x", "x", "x", "x</w>"]
    assert merge("xxxx", XR, lambda t, i: t == 1) == ["xx", "x", "x</w>"]
    assert merge("x", XR, lambda t, i: False) == ["x</w>"]
    # the hash: p = 0 drops nothing, p = 1 everything; the draw depends on (seed, key, word, side, round, position)
    W0 = word_key(5, 7, 0, 0)
    assert not any(hash_drop(W0, thr_of(0.0))(t, i) for t in range(20) for i in range(20))
    assert all(hash_drop(W0, thr_of(1.0))(t, i) for t in range(20) for i in range(20))
    assert len({word_key(5, 7, 0, 0), word_key(5, 7, 0, 1), word_key(5, 7, 1, 0), word_key(5, 8, 0, 0), word_key(6, 7, 0, 0)}) == 5
    assert word_key(5, 7, 3, 1) == mix((mix((mix(5 ^ KEY) + 7 * GOLD) & M64) + 8 * GOLD) & M64)


@pytest.fixture(scope="module")
def host():
    from genz_tokenize_b200 import Tokenize
    t = Tokenize(devices=[])
    return t, Rule(t)


def test_p0_is_the_oracle_bpe(host, oracle):
    t, R = host
    words = [w[:-2] if w.endswith("@@") else w for w in R.enc if w and not re.search(r"\s", w)]
    words += ["xin\n", "chào\n", "ab", "a", "\u0111\u01b0\u1eddng", "</s>", "@@", "</w>", "a" * 300]
    for w in words:
        syms = merge(w, R.ranks, lambda t_, i: False)
        assert "@@ ".join(s for s in syms[:-1]) + ("@@ " if len(syms) > 1 else "") + syms[-1][:-4] == oracle.bpe(w), w
        assert merge(w, R.ranks, hash_drop(word_key(1, 2, 0, 0), 0)) == syms


def test_arguments_rejected(host):
    t, _ = host
    for kw in (dict(padding=False), dict(truncation=False), dict(truncation="longest_first"), dict(max_len=None), dict(max_len=3),
               dict(return_offset=True), dict(return_offsets_mapping=True), dict(bpe_dropout=1.5), dict(bpe_dropout=-0.1),
               dict(bpe_dropout=float("nan"))):
        args = dict(max_len=16, bpe_dropout=0.1)
        args.update(kw)
        with pytest.raises(ValueError):
            t.encode_batch(["a b"], ["c d"], **args)
    for kw in (dict(max_len=3), dict(truncation="only_first"), dict(bpe_dropout=2.0)):
        args = dict(max_len=16, bpe_dropout=0.1)
        args.update(kw)
        with pytest.raises(ValueError):
            t.encode_device(None, None, **args)
    with pytest.raises(ValueError):
        t.encode_batch(["a b"], max_len=16, bpe_dropout=0.1, row_keys=[1, 2])
    with pytest.raises(ValueError):
        t.bpe("xin", dropout=1.01)
    lib = L.load()
    tb = np.frombuffer(b"a b", dtype=np.uint8).copy()
    to = np.array([0, 3], dtype=np.int64)
    enc = L.Encoded()
    call = lambda n, ml, flags, p: lib.genztok_encode_dropout(t._h, tb.ctypes.data, to.ctypes.data, tb.ctypes.data, to.ctypes.data, n, ml, flags, p, 1, None,
                                                             C.byref(enc))
    P = L.DevPlanes()
    P.input_ids = P.attention_mask = P.row_len = 16
    dcall = lambda n, ml, flags, p: lib.genztok_encode_dropout_device(t._h, 0, 16, 16, 3, 16, 16, 3, n, ml, flags, p, 1, None, C.byref(P), None)
    for n, ml, flags, p in ((1, 16, L.WANT_OFFSETS, 0.1), (1, 16, L.WANT_SPANS, 0.1), (1, 16, L.LONGEST_FIRST, 0.1), (1, 16, L.ONLY_SECOND, 0.1),
                            (1, 3, 0, 0.1), (1, L.MAX_LEN_NONE, 0, 0.1), (1, 16, 0, -0.5), (1, 16, 0, 1.5), (1, 16, 0, float("nan")), (-1, 16, 0, 0.1)):
        assert call(n, ml, flags, p) == L.E_INVALID, (n, ml, flags, p)
        assert dcall(n, ml, flags, p) == L.E_INVALID, (n, ml, flags, p)
    assert dcall(1, 16, 0, 0.1) == L.E_NODEVICE                      # valid arguments reach the device check
    assert call(1, 16, L.WANT_TOKEN_TYPE | L.WANT_SEQUENCE_ID, 0.0) == L.E_NODEVICE
    assert call(1, 4, 0, 1.0) == L.E_NODEVICE
    n = C.c_int64()
    assert lib.genztok_bpe_word_dropout(t._h, b"xin", 3, 2.0, 0, 0, None, 0, C.byref(n)) == L.E_INVALID
    assert lib.genztok_bpe_word_dropout(t._h, b"xin", 3, 0.5, 0, 0, None, 0, C.byref(n)) == L.E_NODEVICE


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tok():
    from genz_tokenize_b200 import Tokenize
    return Tokenize(devices=[0])


@pytest.fixture(scope="module")
def rule(tok):
    return Rule(tok)


PLANES = ("input_ids", "attention_mask", "row_len", "token_type_ids", "tt_len", "sequence_id", "seq_len", "row_status")


def same_planes(x, y, what, keys=PLANES):
    for k in keys:
        if k in x or k in y:
            a = x[k].cpu().numpy() if hasattr(x[k], "cpu") else np.asarray(x[k])
            b = y[k].cpu().numpy() if hasattr(y[k], "cpu") else np.asarray(y[k])
            bad = np.argwhere(a != b)
            assert not len(bad), "%s: %s differs first at %s" % (what, k, bad[0])


def assert_rule_rows(got, exp, what):
    from test_windows import as_ids
    for k in ("input_ids", "attention_mask", "row_len"):
        a, b = np.asarray(got[k]), exp[k]
        bad = np.argwhere(a != b)
        assert not len(bad), "%s: %s differs first at %s:\n ours=%s\n rule=%s" % (what, k, bad[0], a[bad[0][0]].tolist(), b[bad[0][0]].tolist())
    if "row_status" in exp:
        assert np.array_equal(got["row_status"], exp["row_status"]), what
        ok = exp["row_status"] == 0
        assert np.array_equal(got["seq_len"][ok], exp["seq_len"][ok]), what
        assert np.array_equal(as_ids(got["token_type_ids"], 0, 2)[ok], exp["token_type_ids"][ok]), what
        assert np.array_equal(got["sequence_id"][ok].astype(np.int64), exp["sequence_id"][ok]), what


WS29 = ["\t", "\n", "\x0b", "\x0c", "\r", "\x1c", "\x1d", "\x1e", "\x1f", " ", "\x85", "\xa0", "\u1680"] + [chr(c) for c in range(0x2000, 0x200b)] + \
       ["\u2028", "\u2029", "\u202f", "\u205f", "\u3000"]


def mixed(seed, n, W, long_rows=None):
    """Singles / pairs around max_len W: noisy text, every one of the 29 whitespace code points, 1,200-byte words, literal <s> / </s>.
    long_rows: only the first long_rows rows keep their 1,200-byte words; later ones are cut to 150 bytes (still merged in global
    memory, and cheaper for the restatement)."""
    from test_truncation import _mixed
    a, b = _mixed(seed, n, W)
    for i in range(0, n, 9):
        ws = WS29[(i // 9) % len(WS29)]
        a[i] = ws.join(a[i].split(" ")) + ws + "xin" + ws
    if long_rows is not None:
        cut = lambda s: " ".join(w[:150] for w in s.split(" "))
        a = a[:long_rows] + [cut(x) for x in a[long_rows:]]
        b = b[:long_rows] + [cut(x) for x in b[long_rows:]]
    return a, b


@gpu
@pytest.mark.parametrize("W", [4, 5, 16, 128, 130, 512])
def test_p0_equals_encode_batch(tok, W):
    a, b = mixed(700 + W, 700, W)
    assert len(WS29) == 29
    for pairs in (None, b):
        ref = tok.encode_batch(a, pairs, max_len=W, sequence_id=True)
        got = tok.encode_batch(a, pairs, max_len=W, sequence_id=True, bpe_dropout=0.0, seed=3)
        same_planes(got, ref, "W=%d pairs=%s" % (W, pairs is not None))
        assert got["real_tokens"] == ref["real_tokens"]


@gpu
def test_p0_pad_token_is_a_vocab_word():
    from golden_util import load_padtt_golden
    from genz_tokenize_b200 import Tokenize
    from genz_tokenize_b200.data import bundled_paths
    from oracle.oracle import Oracle
    v, bp = bundled_paths()
    rng = np.random.default_rng(9)
    for blk in load_padtt_golden() + [{"pad_token": "</s>", "pad_id": 2}]:
        pt = blk["pad_token"]
        t = Tokenize(pad_token=pt, devices=[0])
        words = ["xin", "chào", "sinh_viên", pt, "</s>", "<s>", "<pad>", "hello", "của", "các"]
        mk = lambda n, lo, hi: [" ".join(rng.choice(words, int(rng.integers(lo, hi)))) for _ in range(n)]
        texts, ctx = mk(300, 0, 60), mk(300, 0, 90)
        for W in (13, 48, 128):
            for pairs in (None, ctx):
                got = t.encode_batch(texts, pairs, max_len=W, sequence_id=True, bpe_dropout=0.0)
                ref = t.encode_batch(texts, pairs, max_len=W, sequence_id=True)
                what = "pad %r W=%d pairs=%s" % (pt, W, pairs is not None)
                if pt == "</s>":
                    # the pad is the </s> token: the reference's mask is ids != pad (tokenize.py:148-152), 0 on the framing </s> too,
                    # as the oracle gives it; the fixed pipeline keeps 1 there at some widths
                    same_planes(got, ref, what, tuple(k for k in PLANES if k != "attention_mask"))
                    exp = Oracle(v, bp, [pt, None, None, None, None]).encode_batch(texts, pairs, max_len=W)
                    assert np.array_equal(got["attention_mask"].reshape(-1), exp["mask"]), what
                    continue
                same_planes(got, ref, what)


@gpu
def test_p1_is_the_code_points(tok, rule):
    a, b = mixed(800, 400, 128)
    got = tok.encode_batch(a, b, max_len=128, sequence_id=True, bpe_dropout=1.0, seed=11)
    R = rule
    for d in range(len(a)):
        exp = [R.bos]
        for text, tail in ((a[d], [R.eos, R.eos]), (b[d], [R.eos])):
            ids = []
            for w in re.findall(r"\S+\n?", text):
                ids += [R.enc.get(c + "@@", R.unk) for c in w[:-1]] + [R.enc.get(w[-1], R.unk)]
            exp += ids[:128] + tail
        exp = exp if len(exp) <= 128 else exp[:127] + [R.eos]
        assert got["input_ids"][d, :len(exp)].tolist() == exp, d
        assert got["row_len"][d] == len(exp)


@gpu
@pytest.mark.parametrize("p", [0.05, 0.1, 0.5])
def test_rows_equal_the_restatement(tok, rule, oracle, p):
    for W, n in ((16, 1500), (130, 1000), (512, 300)):
        a, b = mixed(900 + W, n, W, long_rows=16)
        keys = np.random.default_rng(W).integers(-2 ** 63, 2 ** 63 - 1, n, dtype=np.int64)
        for pairs in (None, b):
            got = tok.encode_batch(a, pairs, max_len=W, sequence_id=True, bpe_dropout=p, seed=12345 + W, row_keys=keys)
            assert_rule_rows(got, rule.rows(oracle, a, pairs, W, p, 12345 + W, keys), "p=%g W=%d pairs=%s" % (p, W, pairs is not None))


@gpu
def test_bpe_helper_is_the_first_word_of_a_row(tok, rule):
    words = ["sinh_viên", "công_nghệ", "xxxxxxxxxxxxxxxxxxxx", "nghiêng", "a", "thành_phố_hồ_chí_minh", "đường" * 30, "abcdefghij" * 120]
    for k, w in enumerate(words):
        for p in (0.0, 0.1, 0.5, 1.0):
            key = 1000 * k - 7
            pieces = tok.bpe(w, dropout=p, seed=99, key=key).split("@@ ")
            row = tok.encode_batch([w], max_len=len(w) + 8, bpe_dropout=p, seed=99, row_keys=[key])["input_ids"][0]
            ids = [rule.enc.get(x + "@@", rule.unk) for x in pieces[:-1]] + [rule.enc.get(pieces[-1], rule.unk)]
            assert row[1:1 + len(ids)].tolist() == ids and row[1 + len(ids)] == rule.eos, (w, p)
            syms = merge(w, rule.ranks, hash_drop(word_key(99, key, 0, 0), thr_of(p)))
            assert pieces == [s for s in syms[:-1]] + [syms[-1][:-4]], (w, p)
        assert tok.bpe(w, dropout=0.0) == tok.bpe(w)


def _up(tok, a, dev):
    import torch
    return torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)


@gpu
def test_device_form_equals_host_form_and_does_not_synchronise(tok):
    import torch
    from genz_tokenize_b200.tokenizer import pack_strings
    dev = torch.device("cuda:0")
    a, b = mixed(1000, 3000, 128)
    pa, pb = pack_strings(a), pack_strings(b)
    keys = np.arange(3000, dtype=np.int64) * 3 + 1
    args = lambda: (_up(tok, pa[0], dev), torch.from_numpy(pa[1]).to(dev), _up(tok, pb[0], dev), torch.from_numpy(pb[1]).to(dev))
    side = torch.cuda.Stream(dev)
    for W in (13, 128, 130):
        for p in (0.0, 0.1):
            host = tok.encode_batch(pa, pb, max_len=W, sequence_id=True, bpe_dropout=p, seed=4, row_keys=keys)
            with torch.cuda.stream(side):
                ta, oa, tb, ob = args()
                got = tok.encode_device(ta, oa, tb, ob, max_len=W, sequence_id=True, text_bytes=len(pa[0]), pair_bytes=len(pb[0]),
                                        bpe_dropout=p, seed=4, row_keys=torch.from_numpy(keys).to(dev))
            side.synchronize()
            assert tok.check_errors(dev) == 0
            same_planes(got, host, "W=%d p=%g" % (W, p), tuple(got))
            single = tok.encode_device(ta, oa, max_len=W, text_bytes=len(pa[0]), bpe_dropout=p, seed=4)
            same_planes(single, tok.encode_batch(pa, max_len=W, bpe_dropout=p, seed=4), "single W=%d p=%g" % (W, p), tuple(single))
    # the call is enqueued behind a sleep on the same stream and returns before it ends (no host synchronisation)
    ta, oa, tb, ob = args()
    kw = dict(max_len=128, text_bytes=len(pa[0]), pair_bytes=len(pb[0]), bpe_dropout=0.1, seed=4)
    tok.encode_device(ta, oa, tb, ob, **kw)                          # (buffers sized)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    torch.cuda._sleep(2_000_000_000)
    got = tok.encode_device(ta, oa, tb, ob, **kw)
    returned = torch.cuda.Event()
    returned.record()
    assert not returned.query(), "the call waited for the work before it"
    stop.record()
    torch.cuda.synchronize()
    assert start.elapsed_time(stop) > 100
    same_planes(got, tok.encode_batch(pa, pb, max_len=128, bpe_dropout=0.1, seed=4), "behind a sleep", ("input_ids", "attention_mask", "row_len"))


@gpu
def test_invariance(tok):
    import torch
    from genz_tokenize_b200 import Tokenize
    a, b = mixed(1100, 2000, 64)
    x = tok.encode_batch(a, b, max_len=64, sequence_id=True, bpe_dropout=0.2, seed=8)
    # batch permutation with keys that follow the documents
    perm = np.random.default_rng(1).permutation(len(a))
    y = tok.encode_batch([a[i] for i in perm], [b[i] for i in perm], max_len=64, sequence_id=True, bpe_dropout=0.2, seed=8, row_keys=perm)
    same_planes({k: np.asarray(v)[perm] for k, v in x.items() if k in PLANES}, y, "permutation")
    # chunking, a cold cache, and a normal encode after a dropout call
    small = Tokenize(devices=[0])
    small.set_option("max_chunk_bytes", 8192)
    small.set_option("chunk_rows", 37)
    same_planes(x, small.encode_batch(a, b, max_len=64, sequence_id=True, bpe_dropout=0.2, seed=8), "chunks")
    plain = tok.encode_batch(a, b, max_len=64, sequence_id=True)
    tok.cache_reset()
    same_planes(x, tok.encode_batch(a, b, max_len=64, sequence_id=True, bpe_dropout=0.2, seed=8), "cold cache")
    same_planes(plain, tok.encode_batch(a, b, max_len=64, sequence_id=True), "encode after dropout")
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    multi = Tokenize(devices=list(range(ndev)))
    same_planes(x, multi.encode_batch(a, b, max_len=64, sequence_id=True, bpe_dropout=0.2, seed=8), "devices")


@gpu
def test_seeds(tok):
    a, b = mixed(1200, 1000, 128)
    x = tok.encode_batch(a, b, max_len=128, bpe_dropout=0.1, seed=21)
    same_planes(x, tok.encode_batch(a, b, max_len=128, bpe_dropout=0.1, seed=21), "same seed")
    y = tok.encode_batch(a, b, max_len=128, bpe_dropout=0.1, seed=22)
    assert (x["input_ids"] != y["input_ids"]).any(axis=1).mean() > 0.5
    z = tok.encode_batch(a, b, max_len=128, bpe_dropout=0.1, seed=21, row_keys=np.arange(1000) + 1)
    assert (x["input_ids"] != z["input_ids"]).any(axis=1).mean() > 0.5


@gpu
def test_rates(tok, rule):
    # two-code-point words whose pair has a rank: each occurrence stays merged with probability 1 - p (one draw, round 0, i = 0)
    twos = [w for w in rule.enc if len(w) == 2 and not re.search(r"\s|@", w) and (w[0], w[1] + "</w>") in rule.ranks and
            rule.enc.get(w) is not None][:200]
    assert len(twos) >= 50
    rng = np.random.default_rng(5)
    texts = [" ".join(rng.choice(twos, 100)) for _ in range(1200)]    # 120,000 occurrences
    for p in (0.1, 0.5):
        r = tok.encode_batch(texts, max_len=256, bpe_dropout=p, seed=77)
        unmerged = int(r["row_len"].sum() - 2 * len(texts)) - 120000      # every unmerged occurrence adds one id
        kept = 1 - unmerged / 120000
        assert abs(kept - (1 - p)) < 5 * math.sqrt(p * (1 - p) / 120000), (p, kept)
    # mean pieces per word increase with p
    a, _ = mixed(1300, 2000, 512)
    lens = [int(tok.encode_batch(a, max_len=512, bpe_dropout=p, seed=3)["row_len"].sum()) for p in (0.0, 0.05, 0.2, 0.5, 1.0)]
    assert lens == sorted(lens) and lens[0] < lens[-1], lens


@gpu
def test_decode_is_unchanged(tok):
    from genz_tokenize_b200 import workload
    a, b = workload.generate_hashed(14, 0, 2000, 0, 3, 13), workload.generate_hashed(14, 0, 2000, 1, 3, 13)
    base = tok.encode_batch(a, b, max_len=128, bpe_dropout=0.0)
    got = tok.encode_batch(a, b, max_len=128, bpe_dropout=0.1, seed=2)
    unk = tok._special_ids()[4]
    ok = ~(got["input_ids"] == unk).any(axis=1) & ~(base["input_ids"] == unk).any(axis=1) & (got["row_len"] < 128) & (base["row_len"] < 128)
    assert ok.sum() > 200 and (got["row_len"][ok] > base["row_len"][ok]).any()
    rows = np.nonzero(ok)[0]
    unpadded = lambda r: tok.decode_batch(np.concatenate([r["input_ids"][i, :r["row_len"][i]] for i in rows]),
                                          np.concatenate([[0], np.cumsum(r["row_len"][rows])]))
    assert unpadded(got) == unpadded(base)


@gpu
def test_integration_snippet():
    import os
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "INTEGRATION.md"), encoding="utf-8").read()
    block = text[text.index("BPE-dropout per epoch"):]
    block = block[block.index("```python") + len("```python"):]
    block = block[:block.index("```")]
    env = {}
    exec(compile(block, "INTEGRATION.md", "exec"), env)
    assert env["epochs"][0].shape == env["epochs"][1].shape and not np.array_equal(env["epochs"][0], env["epochs"][1])
    assert np.array_equal(env["same"], env["epochs"][0])


@gpu
def test_offsets_outside_the_text_are_counted():
    import torch
    from genz_tokenize_b200 import Tokenize
    from genz_tokenize_b200.tokenizer import GenztokError
    t = Tokenize(devices=[0])
    dev = torch.device("cuda:0")
    text = torch.zeros(64, dtype=torch.uint8, device=dev)
    text[:20] = torch.tensor(list(b"xin ch\xc3\xa0o sinh_vi\xc3\xaan"[:20]), dtype=torch.uint8)
    # document 1 runs backwards, document 2 past the 20 bytes the call is given: both are counted and get no ids
    off = torch.tensor([0, 8, 4, 4000], dtype=torch.int64, device=dev)
    out = t.encode_device(text, off, max_len=16, text_bytes=20, bpe_dropout=0.1, seed=1)
    torch.cuda.synchronize()
    with pytest.raises(GenztokError, match="inconsistencies"):
        t.check_errors(dev)
    assert out["row_len"].tolist()[1:] == [2, 2]
    assert out["row_len"].tolist()[0] > 2


@gpu
def test_destroy_releases_the_device_buffers():
    import gc
    import torch
    from genz_tokenize_b200 import Tokenize, workload
    dev = torch.device("cuda:0")
    a = workload.generate_hashed(3, 0, 200000, 0, 3, 13)
    d_text = torch.from_numpy(np.concatenate([a[0], np.zeros((-len(a[0])) % 16 + 16, dtype=np.uint8)])).to(dev)
    d_off = torch.from_numpy(a[1]).to(dev)

    def cycle():
        t = Tokenize(devices=[0])
        t.encode_device(d_text, d_off, max_len=64, text_bytes=len(a[0]), bpe_dropout=0.1, seed=1)
        torch.cuda.synchronize()
        del t
        gc.collect()
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info(dev)[0]

    cycle()                                                          # (modules loaded, torch's pools warm)
    free = [cycle() for _ in range(4)]
    # each call holds 8 bytes of scratch per text byte (about 100 MB here) and the streams; a handle that kept them would lose them
    assert free[0] - free[-1] < len(a[0]) * 2, free

