"""Pair truncation strategies (truncation="longest_first" / "only_first" / "only_second") for fixed-layout encodes.

The expected rows are built here from the oracle's untruncated encodes of each side, cut by the Python pair_keep below, then put
through the reference's rules on ids: __padding to max_len, the attention mask (ids != pad), and get_sequence_id + get_token_type
through oracle.sequence_id(ids, True).  pair_keep itself is pinned, on the CPU, to a literal port of the Rust tokenizers' branches.
Argument checks and the host-only handle run on the CPU; everything else on the GPU."""
import ctypes as C

import numpy as np
import pytest

from genz_tokenize_b200 import _lib as L
from test_windows import _streams, as_ids

gpu = pytest.mark.gpu
STRATEGIES = ("longest_first", "only_first", "only_second")


# ---- the rule ------------------------------------------------------------------------------------------------------------
def pair_keep(la, lb, C_, strategy):
    """(la', lb', status 2) -- the closed form of include/genztok.h (csrc/window.cuh: pair_keep)."""
    if la + lb <= C_:
        return la, lb, False
    if strategy == "only_second":
        return (la, C_ - la, False) if la < C_ else (la, lb, True)
    if strategy == "only_first":
        return (C_ - lb, lb, False) if lb < C_ else (la, lb, True)
    s, h = min(la, lb), C_ // 2
    ks = s if s <= h else h
    return (ks, C_ - ks, False) if la <= lb else (C_ - ks, ks, False)


def rust_truncate(la, lb, max_length, strategy):
    """tokenizers::utils::truncation::truncate_encodings for a pair, line by line; max_length is what is left after the added
    tokens.  Returns the kept lengths, or None for Err(SequenceTooShort)."""
    total = la + lb
    if total <= max_length:
        return la, lb
    to_remove = total - max_length
    if strategy == "longest_first":
        n1, n2 = la, lb
        swap = False
        if n1 > n2:
            swap = True
            n1, n2 = n2, n1
        if n1 > max_length:
            n2 = n1
        else:
            n2 = max(n1, max_length - n1)
        if n1 + n2 > max_length:
            n1 = max_length // 2
            n2 = n1 + max_length % 2
        if swap:
            n1, n2 = n2, n1
        return min(la, n1), min(lb, n2)                             # Encoding::truncate(max_len) keeps min(len, max_len)
    target_len = la if strategy == "only_first" else lb
    if target_len > to_remove:
        kept = target_len - to_remove
        return (kept, lb) if strategy == "only_first" else (la, kept)
    return None


def expected_rows(oracle, texts, pairs, W, strategy, specials=(0, 1, 2)):
    """dict of the planes encode_batch(..., truncation=strategy) returns (token types as ids, None as -1)."""
    pad, bos, eos = specials
    A, B = _streams(oracle, texts), _streams(oracle, pairs)
    n = len(A)
    ids = np.full((n, W), pad, dtype=np.int32)
    row_len = np.zeros(n, dtype=np.int32)
    status = np.zeros(n, dtype=np.uint8)
    tt = np.zeros((n, W), dtype=np.int64)
    seq = np.full((n, W), -2, dtype=np.int64)
    seq_len = np.zeros(n, dtype=np.int32)
    for d in range(n):
        a, b = A[d].tolist(), B[d].tolist()
        ka, kb, s2 = pair_keep(len(a), len(b), W - 4, strategy)
        r = [bos] + a[:ka] + [eos, eos] + b[:kb] + [eos]
        if len(r) < W:                                              # __padding (tokenize.py:141-146)
            ids[d, :len(r)] = r
            row_len[d] = len(r)
        else:
            assert s2 or len(r) == W
            ids[d] = r[:W - 1] + [eos]
            row_len[d] = W
        try:
            q = [-1 if v is None else v for v in oracle.sequence_id(ids[d], True)]
        except ValueError:
            status[d] = 1
        else:
            seq_len[d] = len(q)
            seq[d, :len(q)] = q
            tt[d] = (q + [pad] * (W - len(q))) if len(q) < W else q[:W - 1] + [eos]
        if s2:
            status[d] = 2
    return dict(input_ids=ids, attention_mask=(ids != pad).astype(np.uint8), row_len=row_len, token_type_ids=tt, sequence_id=seq,
                seq_len=seq_len, row_status=status)


def assert_rows_equal(got, exp, what, specials=(0, 1, 2)):
    got = {k: (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)) for k, v in got.items()}
    for k in ("input_ids", "attention_mask", "row_len", "row_status"):
        bad = np.argwhere(got[k] != exp[k])
        assert not len(bad), "%s: %s differs first at %s:\n ours=%s\n ref =%s" % (
            what, k, bad[0], got[k][bad[0][0]].tolist() if got[k].ndim > 1 else got[k][bad[0][0]], exp[k][bad[0][0]].tolist() if exp[k].ndim > 1 else exp[k][bad[0][0]])
    ok = exp["row_status"] == 0
    assert np.array_equal(got["seq_len"][ok], exp["seq_len"][ok]), what
    tt = as_ids(got["token_type_ids"], specials[0], specials[2])
    bad = np.argwhere((tt != exp["token_type_ids"]) & ok[:, None])
    assert not len(bad), "%s: token_type_ids differ in row %d:\n ours=%s\n ref =%s\n ids =%s" % (
        what, bad[0][0], tt[bad[0][0]].tolist(), exp["token_type_ids"][bad[0][0]].tolist(), got["input_ids"][bad[0][0]].tolist())
    if "sequence_id" in got:
        assert np.array_equal(got["sequence_id"][ok].astype(np.int64), exp["sequence_id"][ok]), what


PLANES = ("input_ids", "attention_mask", "row_len", "token_type_ids", "tt_len", "sequence_id", "seq_len", "row_status")


def assert_same_planes(x, y, what, rows=None):
    for k in PLANES + ("offset_mapping",):
        if k in x or k in y:
            a, b = np.asarray(x[k]), np.asarray(y[k])
            if rows is not None:
                a, b = a[rows], b[rows]
            assert np.array_equal(a, b), (what, k)


# ---- CPU: the rule, arguments and the host-only handle -------------------------------------------------------------------
def test_closed_form_is_the_rust_rule():
    for C_ in range(0, 41):
        for la in range(0, 41):
            for lb in range(0, 41):
                for s in STRATEGIES:
                    ka, kb, s2 = pair_keep(la, lb, C_, s)
                    r = rust_truncate(la, lb, C_, s)
                    assert (r is None) == s2, (la, lb, C_, s)
                    if r is not None:
                        assert (ka, kb) == r, (la, lb, C_, s, (ka, kb), r)
                        assert ka + kb <= C_ or la + lb <= C_
    # the examples of include/genztok.h and INTEGRATION.md
    assert [pair_keep(a, b, 9, "longest_first")[:2] for a, b in ((3, 20), (20, 3), (10, 10), (20, 10))] == [(3, 6), (6, 3), (4, 5), (5, 4)]


def _host_only():
    from genz_tokenize_b200 import Tokenize
    return Tokenize(devices=[])


def test_strategy_arguments_rejected():
    t = _host_only()
    for kw in (dict(truncation="longest"), dict(truncation="LONGEST_FIRST"), dict(truncation=""),
               dict(truncation="longest_first", padding=False), dict(truncation="only_second", max_len=None),
               dict(truncation="only_first", max_len=3), dict(truncation="longest_first", max_len=0),
               dict(truncation="longest_first", return_offset=True)):
        args = dict(max_len=16)
        args.update(kw)
        with pytest.raises(ValueError):
            t.encode_batch(["a b"], ["c d"], **args)
        with pytest.raises(ValueError):
            t("a b", "c d", **args)
    for kw in (dict(truncation="longest"), dict(truncation="only_first", max_len=3), dict(truncation=False)):
        with pytest.raises(ValueError):
            t.encode_device(None, None, **kw)
    lib = L.load()
    tb = np.frombuffer(b"a b", dtype=np.uint8).copy()
    to = np.array([0, 3], dtype=np.int64)
    enc = L.Encoded()
    call = lambda ml, pad, trunc, flags: lib.genztok_encode(t._h, tb.ctypes.data, to.ctypes.data, tb.ctypes.data, to.ctypes.data, 1, ml, pad, trunc, flags, C.byref(enc))
    for ml, pad, trunc, flags in ((16, 1, 1, L.LONGEST_FIRST | L.ONLY_SECOND), (16, 1, 1, L.ONLY_FIRST | L.ONLY_SECOND), (3, 1, 1, L.ONLY_FIRST),
                                  (L.MAX_LEN_NONE, 1, 1, L.LONGEST_FIRST), (16, 0, 1, L.LONGEST_FIRST), (16, 1, 0, L.ONLY_SECOND),
                                  (16, 1, 1, L.LONGEST_FIRST | L.WANT_SPANS)):
        assert call(ml, pad, trunc, flags) == L.E_INVALID, (ml, pad, trunc, flags)
        assert b"strateg" in lib.genztok_last_error(t._h)
    # valid arguments reach the device check
    for flags in (L.LONGEST_FIRST, L.ONLY_FIRST | L.WANT_OFFSETS, L.ONLY_SECOND):
        assert call(4, 1, 1, flags) == L.E_NODEVICE
    P = L.DevPlanes()
    P.input_ids = P.attention_mask = P.row_len = 16
    dcall = lambda ml, flags, planes: lib.genztok_encode_device(t._h, 0, 16, 16, 3, 16, 16, 3, 1, ml, flags, C.byref(planes), None)
    assert dcall(16, L.LONGEST_FIRST | L.ONLY_FIRST, P) == L.E_INVALID
    assert dcall(3, L.ONLY_SECOND, P) == L.E_INVALID
    assert dcall(16, L.ONLY_SECOND | L.WANT_OFFSETS, P) == L.E_INVALID
    assert dcall(16, L.LONGEST_FIRST, L.DevPlanes()) == L.E_INVALID
    assert dcall(16, L.LONGEST_FIRST, P) == L.E_NODEVICE


def test_strategies_host_only_handle_has_no_cpu_path():
    from genz_tokenize_b200.tokenizer import GenztokError
    t = _host_only()
    for s in STRATEGIES + (True, 1, False, 0):
        with pytest.raises(GenztokError, match="no CPU path"):
            t.encode_batch(["xin chào"], ["hello"], max_len=16, truncation=s)


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tok():
    from genz_tokenize_b200 import Tokenize
    return Tokenize(devices=[0])


def _noisy(seed, n, lo, hi):
    from genz_tokenize_b200 import workload
    return workload.generate(seed, n, lo, hi, 0.05)


def _mixed(seed, n, W):
    """Pairs around max_len W: first longer, second longer, equal, empty sides, 1,200-byte words, literal <s> / </s> words."""
    rng = np.random.default_rng(seed)
    strs = lambda p: [bytes(p[0][p[1][i]:p[1][i + 1]]).decode("utf-8", "surrogatepass") for i in range(len(p[1]) - 1)]
    a, b = strs(_noisy(seed, n, 0, 2 * W + 8)), strs(_noisy(seed + 1, n, 0, 2 * W + 8))
    sw = strs(_noisy(seed + 2, n, 0, max(4, W // 3)))
    out_a, out_b = [], []
    for i in range(n):
        x, y = a[i], b[i]
        k = i % 8
        if k == 1:
            y = sw[i]                                                  # la > lb
        elif k == 2:
            x = sw[i]                                                  # la < lb
        elif k == 3:
            y = x                                                      # la == lb
        elif k == 4:
            x, y = ("", y) if i % 16 < 8 else (x, "")
        elif k == 5:
            long = "".join(rng.choice(list("abcdefghijklmnopqrstuvwxyzàáâãèéêìíòóôõùúýđ"), 1200))
            x, y = (x + " " + long, y) if i % 16 < 8 else (x, long + " " + y)
        elif k == 6:
            words = x.split()
            words.insert(int(rng.integers(0, len(words) + 1)), rng.choice(["</s>", "<s>"]))
            x = " ".join(words)
        elif k == 7:
            words = y.split()
            words.insert(int(rng.integers(0, len(words) + 1)), rng.choice(["</s>", "<s>", "</s> </s>"]))
            y = " ".join(words)
        out_a.append(x)
        out_b.append(y)
    return out_a, out_b


@gpu
def test_rows_that_fit_equal_the_reference_cut(tok):
    from genz_tokenize_b200 import workload
    t, p = workload.generate_hashed(1234, 0, 4000, 0, 3, 13), workload.generate_hashed(1234, 0, 4000, 1, 3, 13)   # bench.py's pairs: all fit
    ref = tok.encode_batch(t, p, max_len=256, sequence_id=True)
    assert (ref["row_len"] < 256).all()
    for s in STRATEGIES:
        got = tok.encode_batch(t, p, max_len=256, sequence_id=True, truncation=s)
        assert_same_planes(got, ref, s)
        assert got["real_tokens"] == ref["real_tokens"]
    # a batch without second texts: every strategy is the reference cut
    ref = tok.encode_batch(t, max_len=8)
    for s in STRATEGIES:
        assert_same_planes(tok.encode_batch(t, max_len=8, truncation=s), ref, s)


@gpu
@pytest.mark.parametrize("W", [4, 5, 13, 128, 130, 512])
def test_overflowing_rows_match_the_rule(tok, oracle, W):
    t, p = _mixed(200 + W, 600, W)
    for s in STRATEGIES:
        exp = expected_rows(oracle, t, p, W, s)
        got = tok.encode_batch(t, p, max_len=W, sequence_id=True, truncation=s)
        assert_rows_equal(got, exp, "%s W=%d" % (s, W))
        assert got["real_tokens"] == int(exp["attention_mask"].sum())
        assert (got["tt_len"] == W).all()
        # status-2 rows hold the reference cut on every plane
        two = exp["row_status"] == 2
        if s != "longest_first" and W >= 13:
            assert two.any(), (s, W)
        if two.any():
            ref = tok.encode_batch(t, p, max_len=W, sequence_id=True)
            assert_same_planes({k: v for k, v in got.items() if k != "row_status"}, {k: v for k, v in ref.items() if k != "row_status"}, s, two)


@gpu
def test_pad_token_is_a_vocab_word(oracle):
    from golden_util import load_padtt_golden
    from genz_tokenize_b200 import Tokenize
    from genz_tokenize_b200.data import bundled_paths
    from oracle.oracle import Oracle
    v, b = bundled_paths()
    rng = np.random.default_rng(7)
    # the golden pad tokens, and a pad that is the </s> token: then the special ids are not distinct and every row takes
    # k_post_rows, which must keep row_status 2
    for blk in load_padtt_golden() + [{"pad_token": "</s>", "pad_id": 2}]:
        pt = blk["pad_token"]
        t = Tokenize(pad_token=pt, devices=[0])
        o = Oracle(v, b, [pt, None, None, None, None])
        words = ["xin", "chào", "sinh_viên", pt, "</s>", "<s>", "<pad>", "hello", "của", "các"]
        mk = lambda n, lo, hi: [" ".join(rng.choice(words, int(rng.integers(lo, hi)))) for _ in range(n)]
        texts, ctx = mk(300, 0, 60), mk(300, 0, 90)
        sp = (blk["pad_id"], 1, 2)
        for W in (13, 48, 128):
            for s in STRATEGIES:
                assert_rows_equal(t.encode_batch(texts, ctx, max_len=W, sequence_id=True, truncation=s), expected_rows(o, texts, ctx, W, s, sp),
                                  "pad %r %s W=%d" % (pt, s, W), sp)


@gpu
def test_offsets_are_the_untruncated_offsets(tok, oracle):
    t, p = _mixed(300, 400, 64)
    ra = tok.encode_batch(t, max_len=None, padding=False, truncation=False, return_offsets_mapping=True)
    rb = tok.encode_batch(p, max_len=None, padding=False, truncation=False, return_offsets_mapping=True)
    side = lambda r, d: r["offset_mapping"][r["row_off"][d] + 1:r["row_off"][d + 1] - 1]
    for W in (13, 64, 130):
        cut = tok.encode_batch(t, p, max_len=W, return_offsets_mapping=True)["offset_mapping"]
        for s in STRATEGIES:
            plain = tok.encode_batch(t, p, max_len=W, sequence_id=True, truncation=s)
            got = tok.encode_batch(t, p, max_len=W, sequence_id=True, truncation=s, return_offsets_mapping=True)
            assert_same_planes({k: v for k, v in got.items() if k != "offset_mapping"}, plain, (s, W))
            om = got["offset_mapping"]
            for d in range(len(t)):
                oa, ob = side(ra, d), side(rb, d)
                ka, kb, s2 = pair_keep(len(oa), len(ob), W - 4, s)
                exp = np.zeros((W, 2), dtype=np.int32)
                if s2:                                                 # the reference cut's row: its offsets as encode_batch gives them
                    assert np.array_equal(om[d], cut[d]), (s, W, d)
                    continue
                exp[1:1 + ka] = oa[:ka]
                exp[ka + 3:ka + 3 + kb] = ob[:kb]
                assert np.array_equal(om[d], exp), (s, W, d)


@gpu
def test_device_form_equals_host_form(tok):
    import torch
    dev = torch.device("cuda:0")
    up = lambda a: torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)
    from genz_tokenize_b200.tokenizer import pack_strings
    t, p = _mixed(400, 3000, 128)
    a, b = pack_strings(t), pack_strings(p)
    side = torch.cuda.Stream(dev)
    for W in (13, 128, 130):
        for s in STRATEGIES:
            host = tok.encode_batch(a, b, max_len=W, sequence_id=True, truncation=s)
            with torch.cuda.stream(side):
                got = tok.encode_device(up(a[0]), torch.from_numpy(a[1]).to(dev), up(b[0]), torch.from_numpy(b[1]).to(dev), max_len=W,
                                        sequence_id=True, text_bytes=len(a[0]), pair_bytes=len(b[0]), truncation=s)
            side.synchronize()
            assert tok.check_errors(dev) == 0
            for k, v in got.items():
                assert np.array_equal(v.cpu().numpy(), host[k]), (W, s, k)


@gpu
def test_chunking_sharding_and_launches(oracle):
    import torch
    from genz_tokenize_b200 import Tokenize
    t, p = _mixed(500, 700, 64)
    base = Tokenize(devices=[0])
    small = Tokenize(devices=[0])
    small.set_option("chunk_rows", 7)
    tiny = Tokenize(devices=[0])
    tiny.set_option("max_chunk_bytes", 8192)
    for s in STRATEGIES:
        x = base.encode_batch(t, p, max_len=64, sequence_id=True, truncation=s, return_offsets_mapping=True)
        for other in (small, tiny):
            y = other.encode_batch(t, p, max_len=64, sequence_id=True, truncation=s, return_offsets_mapping=True)
            assert set(x) == set(y)
            assert_same_planes(x, y, s)
            assert x["real_tokens"] == y["real_tokens"]
    # kernel launches per call (DESIGN.md): 21 per chunk of at most 8,192 pairs, 25 above (the scans of the two streams take
    # three launches each); the same for the device form
    for n, per in ((10, 21), (1000, 21), (9000, 25)):
        a, b = _noisy(51, n, 0, 80), _noisy(52, n, 0, 80)
        base.encode_batch(a, b, max_len=64, truncation="longest_first")
        c0 = base.launch_count()
        base.encode_batch(a, b, max_len=64, truncation="longest_first")
        assert base.launch_count() - c0 == per, (n, base.launch_count() - c0)
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    multi = Tokenize(devices=list(range(ndev)))
    for s in STRATEGIES:
        x = base.encode_batch(t, p, max_len=64, sequence_id=True, truncation=s, return_offsets_mapping=True)
        y = multi.encode_batch(t, p, max_len=64, sequence_id=True, truncation=s, return_offsets_mapping=True)
        assert_same_planes(x, y, s)


@gpu
def test_recycled_planes_after_strategy_rows(tok, oracle):
    # a fixed-layout encode that reuses pooled planes a strategy call held must not trust padding it did not write
    t, p = _noisy(61, 2000, 0, 40), _noisy(62, 2000, 0, 40)
    for _ in range(2):
        r = tok.encode_batch(t, p, max_len=64, truncation="longest_first")
        del r
        ref = tok.encode_batch(t, p, max_len=64)
        exp = oracle.encode_batch(t, p, max_len=64, threads=8)
        assert np.array_equal(ref["input_ids"].reshape(-1), exp["ids"])
        assert np.array_equal(ref["attention_mask"].reshape(-1), exp["mask"])
        del ref


@gpu
def test_call_on_one_pair(tok):
    one = "sinh_viên"
    a, b = " ".join([one] * 10), " ".join(["hello"] * 10)                 # 10 + 10 tokens, W = 13: C = 9
    r = tok(a, b, max_len=13, truncation="longest_first")
    assert r["input_ids"] == [1] + [770] * 4 + [2, 2] + [30469] * 5 + [2]
    assert r["attention_mask"] == [1] * 13
    assert r["sequence_id"] == [0] * 6 + [1] * 7
    assert r["token_type_ids"] == [0] * 6 + [1] * 6 + [2]                  # a row of exactly max_len: the </s> id last (SURVEY A.4)
    r = tok(a, " ".join(["hello"] * 3), max_len=13, truncation="only_first", return_offsets_mapping=True)
    assert r["input_ids"] == [1] + [770] * 6 + [2, 2] + [30469] * 3 + [2]
    assert r["offset_mapping"][:3] == [(0, 0), (0, 10), (11, 21)] and r["offset_mapping"][-1] == (0, 0)
    with pytest.raises(ValueError, match="None is not in list"):       # the reference cut: A fills the row, B is gone
        tok(a, b, max_len=13, truncation=True)
    for s in ("only_second", "only_first"):
        with pytest.raises(ValueError, match=s):
            tok(" ".join([one] * 9) if s == "only_second" else a, " ".join(["hello"] * 9) if s == "only_first" else b, max_len=13, truncation=s)


@gpu
def test_integration_snippet():
    # the sentence-pair snippet of INTEGRATION.md, as written, against the bundled vocab
    import os
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "INTEGRATION.md"), encoding="utf-8").read()
    block = text[text.index("Sentence pairs whose first text is long"):]
    block = block[block.index("```python") + len("```python"):]
    block = block[:block.index("```")]
    env = {}
    exec(compile(block, "INTEGRATION.md", "exec"), env)
    assert env["row"].endswith("</s> </s> trời đẹp </s>") and "trời đẹp" not in env["cut"]
    assert env["status"].tolist() == [2, 0] and env["keep"].tolist() == [False, True]
