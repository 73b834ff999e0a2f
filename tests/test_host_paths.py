"""Host-buffer calls on a handle: every encode_batch and encode_windows part is ordered behind the previous user of its device's
shared work areas, and a part that fails reports its error and gives the result planes back.  Covered here: host calls issued while
device calls still run on another stream, and a document larger than max_chunk_bytes, on one device and on a later device of several."""
import numpy as np
import pytest

from parity_util import assert_matches_oracle

gpu = pytest.mark.gpu


def _noisy(seed, n, lo, hi):
    from genz_tokenize_b200 import workload
    return workload.generate(seed, n, lo, hi, 0.05)


def _with_document(packed, i, doc):
    """The packed batch with document i replaced by `doc` (bytes)."""
    from genz_tokenize_b200 import workload
    from genz_tokenize_b200.tokenizer import pack_strings
    docs = workload.unpack(*packed)
    docs[i] = doc.decode("utf-8")
    return pack_strings(docs)


@gpu
def test_host_calls_wait_for_device_calls_on_another_stream(oracle):
    import ctypes as C
    import torch
    from genz_tokenize_b200 import Tokenize, preprocess, workload
    from genz_tokenize_b200 import _lib as L
    from oracle import oracle as O
    from test_windows import assert_windows_equal, expected_windows
    dev = torch.device("cuda:0")
    up = lambda a: torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)
    tok = Tokenize(devices=[0])
    big = _noisy(71, 220000, 0, 40)                                  # ~40 MB: one chunk under the default 64 MiB, still running below
    assert 16 << 20 < len(big[0]) < 64 << 20
    docs = workload.long_documents(workload.default_wordlist().words, 40, lo=50, hi=900, seed=12)
    small = _noisy(72, 3000, 0, 30)
    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        st = tok._torch_stream(dev)
        # windows step 1 (it reads the number of windows back), then the large fixed-layout encode and windows step 2, not waited for
        W, s = 96, 24
        wt, wo = up(docs[0]), torch.from_numpy(docs[1]).to(dev)
        woff = torch.empty((len(docs[1]),), dtype=torch.int64, device=dev)
        K = C.c_int64()
        assert tok._lib.genztok_encode_windows_device(tok._h, 0, wt.data_ptr(), wo.data_ptr(), len(docs[0]), None, None, 0, len(docs[1]) - 1, W, s, 0,
                                                      woff.data_ptr(), None, None, None, C.byref(K), st) == 0
        K = K.value
        ids = torch.empty((K, W), dtype=torch.int32, device=dev); mask = torch.empty((K, W), dtype=torch.uint8, device=dev)
        rl = torch.empty((K,), dtype=torch.int32, device=dev); wd = torch.empty((K,), dtype=torch.int64, device=dev); ws = torch.empty((K,), dtype=torch.int32, device=dev)
        P = L.DevPlanes(); P.input_ids, P.attention_mask, P.row_len = ids.data_ptr(), mask.data_ptr(), rl.data_ptr()
        bt, bo = up(big[0]), torch.from_numpy(big[1]).to(dev)
        torch.cuda.current_stream(dev).synchronize()                   # (the uploads; from here on nothing waits for the side stream)
        out = tok.encode_device(bt, bo, max_len=64, text_bytes=len(big[0]))
        assert tok._lib.genztok_encode_windows_device(tok._h, 0, wt.data_ptr(), wo.data_ptr(), len(docs[0]), None, None, 0, len(docs[1]) - 1, W, s, 0,
                                                      woff.data_ptr(), C.byref(P), wd.data_ptr(), ws.data_ptr(), None, st) == 0
    # host calls on the same handle, on its own stream, while the side stream may still run
    ragged = tok.encode_batch(small)
    fixed = tok.encode_batch(small, max_len=64)
    win = tok.encode_windows(docs, max_len=128, stride=32)
    prep = preprocess.run_batch(preprocess.REMOVE_HTML, small, tok=tok)
    torch.cuda.synchronize()
    assert_matches_oracle(ragged, oracle.encode_batch(small, None, threads=8), what="ragged host call")
    assert_matches_oracle(fixed, oracle.encode_batch(small, None, max_len=64, threads=8), what="fixed host call")
    assert_windows_equal(win, expected_windows(oracle, docs, None, 128, 32), "windows host call")
    assert prep == O.preprocess(preprocess.REMOVE_HTML, workload.unpack(*small))
    orc = oracle.encode_batch(big, None, max_len=64, threads=8)
    assert np.array_equal(out["input_ids"].cpu().numpy().reshape(-1), orc["ids"])
    assert np.array_equal(out["attention_mask"].cpu().numpy().reshape(-1), orc["mask"])
    exp = expected_windows(oracle, docs, None, W, s)
    assert np.array_equal(woff.cpu().numpy(), exp["window_off"])
    assert np.array_equal(ids.cpu().numpy(), exp["input_ids"]) and np.array_equal(mask.cpu().numpy(), exp["attention_mask"])
    assert np.array_equal(rl.cpu().numpy(), exp["row_len"]) and np.array_equal(wd.cpu().numpy(), exp["overflow_to_sample_mapping"])
    assert tok.check_errors(dev) == 0


def _oversized_fails_then_recovers(tok, oracle, where):
    """A document of 5,000 bytes at row `where` fails every host-buffer encode; the handle then encodes the same shape again.

    Short rows come first, so that the pooled result planes remember that only their first columns hold anything.  The failing
    fixed-layout call takes those planes, and on a handle over several devices the devices without the large document fill
    them with long rows.  The next call of the same shape gets the planes back and must copy every column that can differ."""
    import gc
    from genz_tokenize_b200.tokenizer import GenztokError
    short, long_ = _noisy(81, 500, 0, 3), _noisy(82, 500, 30, 45)
    want = oracle.encode_batch(short, None, max_len=64, threads=8)
    r = tok.encode_batch(short, max_len=64)
    assert_matches_oracle(r, want, what="short rows")
    del r
    gc.collect()
    bad = _with_document(long_, where, b"x" * 5000)
    for call in (lambda: tok.encode_batch(bad, max_len=64), lambda: tok.encode_batch(bad), lambda: tok.encode_windows(bad, max_len=64, stride=8)):
        with pytest.raises(GenztokError, match="larger than max_chunk_bytes"):
            call()
    assert_matches_oracle(tok.encode_batch(short, max_len=64), want, what="short rows after the failures")


@gpu
def test_oversized_document_fails_and_the_handle_recovers(oracle):
    from genz_tokenize_b200 import Tokenize
    tok = Tokenize(devices=[0])
    tok.set_option("max_chunk_bytes", 4096)                            # the smallest it accepts, before the first encode
    _oversized_fails_then_recovers(tok, oracle, 137)


@gpu
def test_oversized_document_on_a_later_device(oracle):
    import torch
    from genz_tokenize_b200 import Tokenize
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs")
    tok = Tokenize(devices=list(range(ndev)))
    tok.set_option("max_chunk_bytes", 4096)
    _oversized_fails_then_recovers(tok, oracle, 499)                  # the last row: in the last device's shard
