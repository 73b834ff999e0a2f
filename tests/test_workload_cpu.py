"""CPU tests of the measurement plumbing: the counter-based workload generator, the plane digest, oracle/_ref."""
import os

import numpy as np
import pytest

from genz_tokenize_b200 import workload


def test_generate_hashed_ranges_are_independent():
    b, o = workload.generate_hashed(1234, 0, 4000, 0, 3, 13, 0.02)
    for lo, hi in ((0, 1), (17, 900), (3999, 4000)):
        sb, so = workload.generate_hashed(1234, lo, hi - lo, 0, 3, 13, 0.02)
        assert bytes(sb) == bytes(b[o[lo]:o[hi]])
        assert np.array_equal(so, o[lo:hi + 1] - o[lo])
    b1, _ = workload.generate_hashed(1234, 0, 4000, 1, 3, 13, 0.02)          # the other side is another text
    assert bytes(b1) != bytes(b)


def test_generate_hashed_has_the_law_of_the_survey():
    """SURVEY.md 8 d2: 3-13 words a sentence sampled in proportion to the vocab counts -> ~50.5 B per sentence, ~8 words."""
    b, o = workload.generate_hashed(1234, 0, 200000, 0, 3, 13, 0.0)
    docs = workload.unpack(b, o)
    k = np.array([len(d.split(" ")) for d in docs])
    assert k.min() == 3 and k.max() == 13 and abs(k.mean() - 8.0) < 0.05
    assert abs(len(b) / len(docs) - 50.5) < 0.5
    words = set(workload.default_wordlist().words)
    assert all(w in words for d in docs[:2000] for w in d.split(" "))


def test_generate_hashed_noise_kinds():
    b, o = workload.generate_hashed(5, 0, 20000, 0, 3, 13, 0.05)
    text = b.tobytes().decode("utf-8")
    assert "\n" in text and "　" in text and "</w>" in text and "@@" in text and " </s> " in text
    words = set(workload.default_wordlist().words)
    unknown = [w for d in workload.unpack(b, o) for w in d.split(" ") if w not in words]
    assert 0.03 < len(unknown) / (8 * 20000) < 0.08


def test_plane_digest_is_order_independent_and_sensitive():
    rng = np.random.default_rng(0)
    n, W = 300, 32
    ids = rng.integers(0, 48000, (n, W)).astype(np.int32)
    mask = (ids % 3 != 0).astype(np.uint8)
    tt = (ids % 2).astype(np.int8)
    d = workload.plane_digest(ids, mask, tt, row0=1000)
    parts = [(0, 100), (100, 250), (250, 300)]
    assert sum(workload.plane_digest(ids[a:b], mask[a:b], tt[a:b], row0=1000 + a) for a, b in parts) % (1 << 64) == d
    ids2 = ids.copy(); ids2[7, 5] ^= 1
    assert workload.plane_digest(ids2, mask, tt, row0=1000) != d
    assert workload.plane_digest(ids, mask, tt, row0=1001) != d
    assert workload.plane_digest(ids[::-1].copy(), mask[::-1].copy(), tt[::-1].copy(), row0=1000) != d    # rows are tied to their index


def test_oracle_ref_recipe_and_oracle_agree_on_the_bench_workload(oracle):
    """oracle/_ref (the unmodified reference, copied there from a reference checkout by oracle/make_ref.py) against the C oracle
    on noisy pairs of the bench workload."""
    from oracle import ref_pool
    if not ref_pool.available():
        pytest.skip("oracle/_ref is absent: run oracle/make_ref.py --ref <reference checkout>")
    n, W = 1500, 40
    ta, tb = workload.generate_hashed(3, 0, n, 0, 3, 13, 0.05), workload.generate_hashed(3, 0, n, 1, 3, 13, 0.05)
    rows = ref_pool.encode_rows_single(workload.unpack(*ta), workload.unpack(*tb), W)
    orc = oracle.encode_batch(ta, tb, max_len=W, threads=4)
    for i, r in enumerate(rows):
        if r is None:
            assert orc["status"][i] == 1
            continue
        assert orc["status"][i] == 0
        assert orc["ids"][orc["ids_off"][i]:orc["ids_off"][i + 1]].tolist() == r["input_ids"], i
        assert orc["tt"][orc["tt_off"][i]:orc["tt_off"][i + 1]].tolist() == r["token_type_ids"], i


def test_bench_dump_outputs_is_a_fixed_sample_of_the_planes(tmp_path):
    """bench.py --dump-outputs: the same rows every run, their values as float32, the global pair index beside them; the
    full-size dump ([DUMP_ROWS, 256] for three planes plus three per-row arrays and the index) stays under 64 MB."""
    import torch
    import bench
    rng = np.random.default_rng(1)
    m, W = 5000, 64
    planes = {"input_ids": torch.from_numpy(rng.integers(0, 48423, (m, W)).astype(np.int32)),
              "attention_mask": torch.from_numpy(rng.integers(0, 2, (m, W)).astype(np.uint8)),
              "row_status": torch.from_numpy(rng.integers(0, 2, m).astype(np.uint8))}
    for d in ("a", "b"):
        bench.dump_outputs(planes, 7000, str(tmp_path / d), max_rows=300)
    idx = np.load(tmp_path / "a" / "pair_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 300 and (np.diff(idx) > 0).all() and idx[0] >= 7000 and idx[-1] < 7000 + m
    rows = idx.astype(np.int64) - 7000
    for name, plane in planes.items():
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, b)
        assert np.array_equal(a, plane.numpy()[rows].astype(np.float32)), name
    assert bench.DUMP_ROWS * (3 * bench.MAX_LEN * 4 + 3 * 4 + 8) < 64e6


def test_custom_model_builder_roundtrip(tmp_path, oracle):
    from oracle.oracle import Oracle
    vp, mp, words = workload.build_custom_model(str(tmp_path), n_words=300, seed=3)
    o = Oracle(vp, mp)
    b, off = workload.long_documents(words, 4, lo=50, hi=80)
    r = o.encode_batch((b, off), None, max_len=4096)
    docs = workload.unpack(b, off)
    for i, d in enumerate(docs):
        ids = r["ids"][r["ids_off"][i]:r["ids_off"][i + 1]]
        nt = int(r["mask"][r["ids_off"][i]:r["ids_off"][i + 1]].sum())
        assert nt >= len(d.split(" ")) + 2 and ids[0] == 1 and ids[nt - 1] == 2
        assert (ids[1:nt - 1] != 4).mean() > 0.4                                                      # merges of the custom table apply
