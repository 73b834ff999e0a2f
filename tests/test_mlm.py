"""Masked-language-model inputs and labels: Tokenize.mlm_mask.

The expected values come from a numpy restatement of the semantics stated in include/genztok.h, built on workload._mix64 and the
handle's decoder and special ids; a scalar form in plain Python integers pins the restatement's hashes.  The restatement and the
argument checks run on the CPU; everything else on the GPU."""
import math

import numpy as np
import pytest

from genz_tokenize_b200 import _lib as L
from genz_tokenize_b200.workload import _mix64

gpu = pytest.mark.gpu
GOLD, KEY = 0x9E3779B97F4A7C15, 0x6D6C6D5F6D61736B
M64 = 2 ** 64 - 1
U = np.uint64


# ---- the restatement ----------------------------------------------------------------------------------------------------------
def tables(tok):
    """(n_ids, continuation flags [n_ids], special ids, repl) of a handle."""
    dec = tok.decoder
    n_ids = max(dec) + 1
    cont = np.zeros(n_ids, dtype=bool)
    for i, s in dec.items():
        cont[i] = s.endswith("@@")
    sp = list(tok._special_ids())
    repl = np.array(sorted(i for i in dec if i not in sp), dtype=np.int64)
    return n_ids, cont, sp, repl


def groups(ids, T, whole_word):
    """g(j) per column: j, or the start of j's word (the column after the last non-continuation id)."""
    n_ids, cont, _, _ = T
    ids = np.asarray(ids, dtype=np.int64)
    n, W = ids.shape
    j = np.broadcast_to(np.arange(W), (n, W))
    if not whole_word:
        return j.copy()
    inr = (ids >= 0) & (ids < n_ids)
    c = np.zeros((n, W), dtype=bool)
    c[inr] = cont[ids[inr]]
    start = np.ones((n, W), dtype=bool)
    start[:, 1:] = ~c[:, :-1]
    return np.maximum.accumulate(np.where(start, j, 0), axis=1)


def ref_mlm(ids, T, seed, p=0.15, a=0.8, b=0.1, whole_word=False, keys=None):
    n_ids, _, sp, repl = T
    ids = np.asarray(ids, dtype=np.int64)
    n, W = ids.shape
    elig = (ids >= 0) & (ids < n_ids) & ~np.isin(ids, sp)
    g = groups(ids, T, whole_word).astype(U)
    j = np.arange(W, dtype=U)[None, :]
    k = np.arange(n, dtype=np.int64) if keys is None else np.asarray(keys, dtype=np.int64)
    s0 = _mix64(np.array([(seed & M64) ^ KEY], dtype=U))[0]
    R = _mix64(s0 + k.view(U) * U(GOLD))[:, None]
    t_sel, t_m, t_mr = math.floor(p * 2 ** 32), math.floor(a * 2 ** 32), math.floor((a + b) * 2 ** 32)
    sel = elig & ((_mix64(R + (U(2) * g + U(1)) * U(GOLD)) >> U(32)) < U(t_sel))
    v = _mix64(R + (U(2) * j + U(2)) * U(GOLD))
    u = v >> U(32)
    out = ids.copy()
    out[sel & (u < U(t_m))] = sp[3]
    rnd = sel & (u >= U(t_m)) & (u < U(t_mr))
    if rnd.any():
        out[rnd] = repl[(((v[rnd] & U(0xFFFFFFFF)) * U(len(repl))) >> U(32)).astype(np.int64)]
    labels = np.where(sel, ids, -100).astype(np.int64)
    return out.astype(np.int32), labels


def scalar_row(row, T, seed, p, a, b, whole_word, key):
    """One row in plain Python integers, literally as include/genztok.h states it."""
    n_ids, cont, sp, repl = T

    def mix(x):
        x ^= x >> 30; x = (x * 0xBF58476D1CE4E5B9) & M64; x ^= x >> 27; x = (x * 0x94D049BB133111EB) & M64; x ^= x >> 31
        return x

    R = mix((mix(seed ^ KEY) + (key & M64) * GOLD) & M64)
    out, lab = list(row), [-100] * len(row)
    for j, x in enumerate(row):
        if not (0 <= x < n_ids and x not in sp):
            continue
        g = j
        while whole_word and g > 0 and 0 <= row[g - 1] < n_ids and cont[row[g - 1]]:
            g -= 1
        if (mix((R + (2 * g + 1) * GOLD) & M64) >> 32) >= math.floor(p * 2 ** 32):
            continue
        v = mix((R + (2 * j + 2) * GOLD) & M64)
        if v >> 32 < math.floor(a * 2 ** 32):
            out[j] = sp[3]
        elif v >> 32 < math.floor((a + b) * 2 ** 32):
            out[j] = int(repl[((v & 0xFFFFFFFF) * len(repl)) >> 32])
        lab[j] = x
    return out, lab


# ---- CPU: the restatement on hand-worked rows ------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host():
    from genz_tokenize_b200 import Tokenize
    t = Tokenize(devices=[])
    return t, tables(t)


def hand_rows(t, T):
    """<s> w1@@ w2@@ w3 x </s> <pad> <pad>: a three-piece word and a one-piece word; <s> <mask> y1@@ <unk> -1 n_ids </s> w: an
    existing mask, a continuation into <unk>, out-of-range ids; x w1@@ w2@@ </s>: a word cut by truncation runs into </s>."""
    n_ids, cont, sp, repl = T
    pad, bos, eos, msk, unk = sp
    cids = [int(i) for i in repl if cont[i]]
    wids = [int(i) for i in repl if not cont[i]]
    c1, c2, c3, w1, w2 = cids[10], cids[20], cids[30], wids[10], wids[20]
    return np.array([[bos, c1, c2, w1, w2, eos, pad, pad],
                     [bos, msk, c3, unk, -1, n_ids, eos, w1],
                     [w2, c1, c2, eos, pad, pad, pad, pad]], dtype=np.int32)


def test_restatement_hand_worked_rows(host):
    t, T = host
    ids = hand_rows(t, T)
    n_ids, cont, sp, repl = T
    pad, bos, eos, msk, unk = sp
    assert groups(ids, T, False).tolist() == [list(range(8))] * 3
    assert groups(ids, T, True).tolist() == [[0, 1, 1, 1, 4, 5, 6, 7],        # w1@@ w2@@ w3 is one word
                                            [0, 1, 2, 2, 4, 5, 6, 7],         # y1@@ <unk>: <unk> joins the word (and is not eligible)
                                            [0, 1, 1, 1, 4, 5, 6, 7]]         # the truncated word runs into </s>
    elig = np.array([[0, 1, 1, 1, 1, 0, 0, 0], [0, 0, 1, 0, 0, 0, 0, 1], [1, 1, 1, 0, 0, 0, 0, 0]], dtype=bool)
    for ww in (False, True):
        out, lab = ref_mlm(ids, T, 5, p=1.0, a=1.0, b=0.0, whole_word=ww)   # everything eligible becomes <mask>
        assert np.array_equal(out, np.where(elig, msk, ids)) and np.array_equal(lab, np.where(elig, ids, -100))
        out, lab = ref_mlm(ids, T, 5, p=1.0, a=0.0, b=0.0, whole_word=ww)   # selected, kept, labelled
        assert np.array_equal(out, ids) and np.array_equal(lab, np.where(elig, ids, -100))
        out, lab = ref_mlm(ids, T, 5, p=0.0, whole_word=ww)
        assert np.array_equal(out, ids) and (lab == -100).all()
        out, lab = ref_mlm(ids, T, 5, p=1.0, a=0.0, b=1.0, whole_word=ww)   # random ids, never special
        assert np.isin(out[elig], repl).all() and not np.isin(out[elig], sp).any() and np.array_equal(out[~elig], ids[~elig])
    # whole words share the decision: over many seeds the three pieces of row 0 are selected together or not at all
    seen = set()
    for seed in range(200):
        _, lab = ref_mlm(ids, T, seed, p=0.5, whole_word=True)
        s = lab[0, 1:4] != -100
        assert s.all() or not s.any()
        seen.add(bool(s[0]))
    assert seen == {False, True}


def test_restatement_equals_scalar_form(host):
    t, T = host
    rng = np.random.default_rng(1)
    n_ids, cont, sp, repl = T
    ids = np.concatenate([hand_rows(t, T), rng.choice(np.concatenate([repl[cont[repl]][:50], repl[:50], sp, [-1, n_ids, n_ids + 7]]),
                                                      size=(20, 8))]).astype(np.int32)
    keys = rng.integers(-2 ** 62, 2 ** 62, size=len(ids))
    for (p, a, b) in [(0.15, 0.8, 0.1), (0.6, 0.5, 0.3), (1.0, 0.0, 1.0), (0.9, 1.0, 0.0)]:
        for ww in (False, True):
            for seed in (0, 2 ** 64 - 1, 12345):
                out, lab = ref_mlm(ids, T, seed, p, a, b, ww, keys)
                for r in range(len(ids)):
                    so, sl = scalar_row([int(x) for x in ids[r]], T, seed, p, a, b, ww, int(keys[r]))
                    assert out[r].tolist() == so and lab[r].tolist() == sl, (p, a, b, ww, seed, r)


def test_argument_checks_host_only_handle(host):
    from genz_tokenize_b200.tokenizer import GenztokError
    t, _ = host
    lib = L.load()
    buf = np.zeros(4096, dtype=np.uint8)
    p, q = buf.ctypes.data, buf.ctypes.data + 1024                         # stand for device pointers: nothing is launched

    def call(**kw):
        a = dict(ids=p, n=4, W=16, keys=None, seed=1, prob=0.15, a=0.8, b=0.1, ww=0, out=q, lab=q + 512)
        a.update(kw)
        return lib.genztok_mlm_mask_device(t._h, 0, a["ids"], a["n"], a["W"], a["keys"], a["seed"], a["prob"], a["a"], a["b"], a["ww"],
                                           a["out"], a["lab"], None)

    for kw, msg in [(dict(prob=-0.1), b"finite and in [0, 1]"), (dict(prob=float("nan")), b"finite"), (dict(a=1.5), b"in [0, 1]"),
                    (dict(b=float("inf")), b"finite"), (dict(a=0.7, b=0.4), b"<= 1"), (dict(n=-1), b"n >= 0"), (dict(W=0), b"width >= 1"),
                    (dict(ids=None), b"required"), (dict(out=None), b"required"), (dict(lab=None), b"required"),
                    (dict(out=p), b"must not overwrite")]:
        assert call(**kw) == L.E_INVALID, kw
        assert msg in lib.genztok_last_error(t._h), (kw, lib.genztok_last_error(t._h))
    assert call(n=0, ids=None, out=None, lab=None) == L.E_NODEVICE        # nothing to do, but the slot is still checked
    assert call() == L.E_NODEVICE
    assert call(a=0.5, b=0.5, ww=1, keys=p) == L.E_NODEVICE
    assert b"no such device" in lib.genztok_last_error(t._h)
    with pytest.raises(GenztokError, match="no CPU path"):
        t.mlm_mask(np.zeros((2, 8), np.int32), seed=1)
    with pytest.raises(TypeError):
        t.mlm_mask(np.zeros((2, 8), np.int32))                              # no default seed: no static masking by accident
    for bad in (np.zeros((2, 8), np.float32), np.zeros((2, 8), bool)):
        with pytest.raises(TypeError, match="integers"):
            t.mlm_mask(bad, seed=1)                                         # a float or bool plane is an error, not a silent cast


def test_random_replacement_needs_a_vocab_id(tmp_path):
    from genz_tokenize_b200 import Tokenize
    vp, mp = tmp_path / "v.txt", tmp_path / "m.codes"
    vp.write_text("<s> 1\n</s> 1\n")                                         # only special strings: nothing to draw from
    mp.write_text("#version: 0.2\n")
    t = Tokenize.fromFile(str(vp), str(mp), devices=[])
    lib = L.load()
    buf = np.zeros(1024, dtype=np.uint8)
    call = lambda b: lib.genztok_mlm_mask_device(t._h, 0, buf.ctypes.data, 1, 4, None, 1, 0.15, 0.8, b, 0, buf.ctypes.data + 64, buf.ctypes.data + 128, None)
    assert call(0.1) == L.E_INVALID and b"no id to draw" in lib.genztok_last_error(t._h)
    assert call(0.0) == L.E_NODEVICE


# ---- GPU --------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tok():
    from genz_tokenize_b200 import Tokenize
    return Tokenize(devices=[0])


PAB = [(0.0, 0.8, 0.1), (0.15, 0.8, 0.1), (1.0, 0.8, 0.1), (0.15, 1.0, 0.0), (1.0, 0.0, 1.0), (1.0, 0.0, 0.0)]


def check_plane(tok, T, ids, what, seeds=(3,), pab=PAB, keys=None):
    """The device result equals the restatement (both modes) and holds the invariants; returns the number of comparisons."""
    import torch
    dev = torch.device("cuda:0")
    d = ids if isinstance(ids, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(ids)).to(dev)
    h = d.cpu().numpy()
    n_ids, cont, sp, repl = T
    elig = (h >= 0) & (h < n_ids) & ~np.isin(h, sp)
    for seed in seeds:
        for p, a, b in pab:
            for ww in (False, True):
                out, lab = tok.mlm_mask(d, seed, mlm_probability=p, whole_word=ww, mask_replace_prob=a, random_replace_prob=b, row_keys=keys)
                assert out.dtype == torch.int32 and lab.dtype == torch.int64 and out.device == d.device
                out, lab = out.cpu().numpy(), lab.cpu().numpy()
                eo, el = ref_mlm(h, T, seed, p, a, b, ww, None if keys is None else keys.cpu().numpy())
                bad = np.argwhere((out != eo) | (lab != el))
                assert not len(bad), "%s p=%g a=%g b=%g ww=%d: at %s ours (%d, %d), ref (%d, %d)" % (
                    what, p, a, b, ww, tuple(bad[0]), out[tuple(bad[0])], lab[tuple(bad[0])], eo[tuple(bad[0])], el[tuple(bad[0])])
                assert (lab[~elig] == -100).all()                           # no special or out-of-range column is labelled
                assert np.array_equal(out[lab == -100], h[lab == -100])
                assert np.array_equal(lab[lab != -100], h[lab != -100])
                if ww:                                                      # every eligible column of a group shares the decision
                    g = groups(h, T, True)
                    s = (lab != -100)
                    rows = np.repeat(np.arange(len(h)), h.shape[1]).reshape(h.shape)
                    first = {}
                    for r_, g_, s_ in zip(rows[elig], g[elig], s[elig]):
                        assert first.setdefault((r_, g_), s_) == s_
    assert np.array_equal(d.cpu().numpy(), h)                               # the input is not modified
    assert tok.check_errors() == 0


@gpu
@pytest.mark.parametrize("W", [16, 128, 512])
def test_encode_batch_planes(tok, W):
    from test_offsets import noisy_rows
    T = tables(tok)
    texts = noisy_rows(300 + W, 120)
    e = tok.encode_batch(texts, max_len=W)
    check_plane(tok, T, e["input_ids"], "singles W=%d" % W)
    ep = tok.encode_batch(texts[:60], texts[60:], max_len=W)
    check_plane(tok, T, ep["input_ids"], "pairs W=%d" % W, pab=PAB[1:3])


@gpu
def test_window_planes_noisy_text(tok):
    from genz_tokenize_b200 import workload
    from test_offsets import unpack
    T = tables(tok)
    texts = unpack(workload.generate(11, 200, 20, 400, noise=0.3))
    texts[0] = "đường</s> sinh_viên@@ x\ny @@ <unk> <mask> " * 20
    for W, s in [(130, 40), (64, 0), (512, 100)]:
        w = tok.encode_windows(texts, max_len=W, stride=s)
        assert len(w["input_ids"]) > len(texts)
        check_plane(tok, T, w["input_ids"], "windows W=%d s=%d" % (W, s), pab=PAB[1:3])


@gpu
def test_custom_and_moved_specials(tok):
    from genz_tokenize_b200 import Tokenize
    from test_offsets import noisy_rows
    texts = noisy_rows(5, 80) + ["[MASK] p@@ ab [UNK] [PAD]"]
    for sp in (["[PAD]", "[CLS]", "[SEP]", "[MASK]", "[UNK]"], ["p@@", "<s>", "</s>", "ab", "<unk>"]):
        t = Tokenize(*sp)
        T = tables(t)
        ids = t.encode_batch(texts, max_len=48)["input_ids"].copy()                # (result planes are recycled: never write into one)
        if sp[0] == "p@@":
            # vocab.txt holds "p@@" and "ab": the pad and mask ids moved (SURVEY A.6) and ids 0 and 3 left the decoder; such ids are
            # eligible, never continue, and a "p@@" piece in the text is the pad id (not a continuation)
            assert t._special_ids()[0] != 0 and t._special_ids()[3] != 3 and 0 not in t.decoder and 3 not in t.decoder
            ids[:, -6:] = [0, 3, 0, t._special_ids()[0], 3, 5]
        check_plane(t, T, ids, "specials %s" % sp[0], pab=PAB[1:3] + PAB[4:5])


@gpu
def test_odd_widths_and_unaligned_planes(tok):
    import torch
    from test_offsets import noisy_rows
    T = tables(tok)
    dev = torch.device("cuda:0")
    texts = noisy_rows(9, 100)
    for W in (37, 130, 1):
        check_plane(tok, T, tok.encode_batch(texts, max_len=W)["input_ids"], "W=%d" % W, pab=PAB[1:3])
    ids = torch.from_numpy(tok.encode_batch(texts, max_len=64)["input_ids"]).to(dev)
    buf = torch.empty(ids.numel() + 1, dtype=torch.int32, device=dev)
    un = buf[1:].view(ids.shape)
    un.copy_(ids)
    assert un.data_ptr() % 16 == 4
    check_plane(tok, T, un, "unaligned", pab=PAB[1:2])
    check_plane(tok, T, ids[:, 4:], "column slice", pab=PAB[1:2])           # a strided view goes through .contiguous()


@gpu
def test_row_keys_seeds_and_repeats(tok):
    import torch
    from test_offsets import noisy_rows
    T = tables(tok)
    dev = torch.device("cuda:0")
    ids = torch.from_numpy(tok.encode_batch(noisy_rows(21, 200), max_len=128)["input_ids"]).to(dev)
    keys = torch.arange(1000, 1200, dtype=torch.int64, device=dev) * 7919 - 10 ** 6
    check_plane(tok, T, ids, "keys", pab=PAB[1:2], keys=keys)
    perm = torch.randperm(200, generator=torch.Generator().manual_seed(0)).to(dev)
    for ww in (False, True):
        o1, l1 = tok.mlm_mask(ids, 42, whole_word=ww, row_keys=keys)
        o2, l2 = tok.mlm_mask(ids[perm], 42, whole_word=ww, row_keys=keys[perm])   # masking does not depend on batch order
        assert torch.equal(o1[perm], o2) and torch.equal(l1[perm], l2)
        o3, l3 = tok.mlm_mask(ids, 42, whole_word=ww, row_keys=keys)
        assert torch.equal(o1, o3) and torch.equal(l1, l3)                   # bit-identical from run to run
        o4, l4 = tok.mlm_mask(ids, 43, whole_word=ww, row_keys=keys)
        assert not torch.equal(l1, l4)                                        # another seed, another mask
        o5, l5 = tok.mlm_mask(ids.long(), 42, whole_word=ww, row_keys=keys.cpu().numpy())   # int64 ids, numpy keys
        assert torch.equal(o1, o5) and torch.equal(l1, l5)
    # int64 ids outside the int32 range are never eligible and come back clamped; float planes are refused
    wide = ids.long()
    wide[:, 5] = 2 ** 40
    wide[:, 6] = -2 ** 40
    o6, l6 = tok.mlm_mask(wide, 42, mlm_probability=1.0)
    assert (o6[:, 5] == 2 ** 31 - 1).all() and (o6[:, 6] == -1).all() and (l6[:, 5:7] == -100).all()
    ho, hl = tok.mlm_mask(wide.cpu().numpy(), 42, mlm_probability=1.0)
    assert np.array_equal(ho, o6.cpu().numpy()) and np.array_equal(hl, l6.cpu().numpy())
    with pytest.raises(TypeError, match="integers"):
        tok.mlm_mask(ids.float(), 42)


@gpu
def test_rates(tok):
    import torch
    T = tables(tok)
    n_ids, cont, sp, repl = T
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(5)
    r = torch.from_numpy(repl).to(dev)
    ids = r[torch.randint(0, len(repl), (8192, 512), generator=g, device=dev)].to(torch.int32)   # 4 M eligible columns
    N = ids.numel()
    p = 0.15
    out, lab = tok.mlm_mask(ids, 2024, mlm_probability=p)
    sel = lab != -100
    S = int(sel.sum())
    assert abs(S - N * p) <= 6 * math.sqrt(N * p * (1 - p)), S
    nm = int((out[sel] == sp[3]).sum())
    nk = int((out[sel] == ids[sel]).sum())
    for cnt, q in ((nm, 0.8), (S - nm - nk, 0.1), (nk, 0.1)):
        # a random draw can equal the original id; the kept share absorbs those (about 1 / len(repl) of the random ones)
        assert abs(cnt - S * q) <= 6 * math.sqrt(S * q * (1 - q)) + S * 0.1 / len(repl) + 1, (cnt, S, q)
    # random ids: only repl, every id of repl drawn, none far from uniform
    out, lab = tok.mlm_mask(ids, 7, mlm_probability=1.0, mask_replace_prob=0.0, random_replace_prob=1.0)
    assert torch.equal(lab, ids.long())
    c = torch.bincount(out.reshape(-1).long(), minlength=n_ids).cpu().numpy()
    assert c[np.setdiff1d(np.arange(n_ids), repl)].sum() == 0
    lam = N / len(repl)
    assert c[repl].min() > 0 and np.abs(c[repl] - lam).max() <= 6 * math.sqrt(lam * (1 - 1 / len(repl))), (c[repl].min(), c[repl].max(), lam)
    # whole words: selected groups among all groups
    out, lab = tok.mlm_mask(ids, 2024, mlm_probability=p, whole_word=True)
    h, s = ids.cpu().numpy(), (lab != -100).cpu().numpy()
    gs = np.zeros(h.shape, dtype=bool)
    gs[:, 0] = True
    gs[:, 1:] = ~cont[h[:, :-1]]
    G, SG = int(gs.sum()), int(s[gs].sum())
    assert abs(SG - G * p) <= 6 * math.sqrt(G * p * (1 - p)), (SG, G)
    assert tok.check_errors() == 0


@gpu
def test_host_form_launches_and_empty(tok):
    import torch
    from test_offsets import noisy_rows
    T = tables(tok)
    dev = torch.device("cuda:0")
    e = tok.encode_batch(noisy_rows(4, 64), max_len=96)
    d = torch.from_numpy(e["input_ids"]).to(dev)
    for ww in (False, True):
        ho, hl = tok.mlm_mask(e["input_ids"], 9, whole_word=ww)
        assert isinstance(ho, np.ndarray) and ho.dtype == np.int32 and hl.dtype == np.int64
        n0 = tok.launch_count()
        do, dl = tok.mlm_mask(d, 9, whole_word=ww)
        assert tok.launch_count() - n0 == 1
        assert np.array_equal(ho, do.cpu().numpy()) and np.array_equal(hl, dl.cpu().numpy())
        eo, el = ref_mlm(e["input_ids"], T, 9, whole_word=ww)
        assert np.array_equal(ho, eo) and np.array_equal(hl, el)
    n0 = tok.launch_count()
    o, l = tok.mlm_mask(torch.zeros((0, 16), dtype=torch.int32, device=dev), 1)
    assert tok.launch_count() == n0 and o.shape == (0, 16) and l.shape == (0, 16)
    # a DataCollection-style batch on another stream
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        o2, l2 = tok.mlm_mask(d, 9)
    s.synchronize()
    assert torch.equal(o2, tok.mlm_mask(d, 9)[0])
    assert tok.check_errors() == 0


@gpu
def test_integration_snippet():
    # the MLM snippet of INTEGRATION.md, as written, against the bundled vocab
    import os
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "INTEGRATION.md"), encoding="utf-8").read()
    block = text[text.index("Masked language modelling on the GPU"):]
    block = block[block.index("```python") + len("```python"):]
    block = block[:block.index("```")]
    env = {}
    exec(compile(block, "INTEGRATION.md", "exec"), env)
    assert env["steps"] == 9 and env["masked_tokens"] > 0
