"""Extractive QA on one GPU: qa_labels (bytes and characters) and qa_best_spans over the windows of question + context pairs, with
the host-side baselines on the same windows.
    python tools/qa_case.py OUT_DIR        -> OUT_DIR/qa_case.json
Workloads: the 4,096 question + context pairs of tools/windows_case.py (5-20 word questions, 300-1,500 word contexts) and 32,768
pairs from the same generator, at max_len=384 / stride=128.  Answers are random word-aligned spans of 1-8 words, given both as
bytes and as Python str indices.  Logits are random float32 normals.  Baselines: the numpy per-window labelling loop INTEGRATION.md
gave before this change, and a numpy per-window best-span search (both timed on a subset of the windows and scaled, noted in the
file)."""
import json, os, re, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from genz_tokenize_b200 import Tokenize, workload

out_dir = sys.argv[1]
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda:0")
WORD = re.compile(r"\S+\n?")
W, STRIDE, L_ = 384, 128, 30


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"nvidia_smi": q.stdout.strip(), "torch_name": torch.cuda.get_device_name(0)}


def hbm_copy_gbs():
    """Measured device-to-device copy bandwidth (read + write bytes), 2 GiB buffers."""
    a = torch.empty((1 << 31,), dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    del a, b
    torch.cuda.empty_cache()
    return 2 * (1 << 31) / (ms * 1e-3) / 1e9


def timed(fn, reps):
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def answers_for(ctx_strs, seed):
    rng = np.random.default_rng(seed)
    by, ch = [], []
    for t in ctx_strs:
        ms = list(WORD.finditer(t))
        i = int(rng.integers(0, len(ms)))
        j = min(len(ms) - 1, i + int(rng.integers(0, 8)))
        k0, k1 = ms[i].start(), ms[j].start() + len(ms[j].group(0).rstrip("\n"))
        ch.append((k0, k1))
        by.append((len(t[:k0].encode("utf-8", "surrogatepass")), len(t[:k1].encode("utf-8", "surrogatepass"))))
    return np.array(by, dtype=np.int64), np.array(ch, dtype=np.int64)


def numpy_labels(om, tt, doc, answers, rows):
    """The recipe INTEGRATION.md gave: a numpy pass per window."""
    st = np.zeros(len(rows), dtype=np.int64); en = np.zeros(len(rows), dtype=np.int64)
    for k, i in enumerate(rows):
        a0, a1 = answers[doc[i]]
        ctx = (tt[i] == 1) & (om[i, :, 1] > 0)
        inside = ctx & (om[i, :, 0] < a1) & (om[i, :, 1] > a0)
        cols = np.flatnonzero(inside)
        if len(cols) and om[i, cols[0], 0] <= a0 and om[i, cols[-1], 1] >= a1:
            st[k], en[k] = cols[0], cols[-1]
    return st, en


def numpy_spans(S, E, om, tt, rows):
    """A numpy best-span search per window: the [c, c] score matrix of the context columns, masked to e >= s, e - s < L."""
    out = []
    for i in rows:
        cols = np.flatnonzero((tt[i] == 1) & (om[i, :, 1] > 0))
        if not len(cols):
            continue
        sc = S[i, cols][:, None] + E[i, cols][None, :]
        d = cols[None, :] - cols[:, None]
        sc = np.where((d >= 0) & (d < L_), sc, -np.inf)
        a = int(np.argmax(sc))
        out.append((float(sc.flat[a]), a // len(cols), a % len(cols)))
    return out


def case(name, tok, q, ctx, bw):
    ctx_strs = [bytes(ctx[0][ctx[1][i]:ctx[1][i + 1]]).decode("utf-8", "surrogatepass") for i in range(len(ctx[1]) - 1)]
    n = len(ctx_strs)
    up = lambda a: torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)
    dq, dc = (up(q[0]), torch.from_numpy(q[1]).to(dev)), (up(ctx[0]), torch.from_numpy(ctx[1]).to(dev))
    w = tok.encode_windows_device(dq[0], dq[1], dc[0], dc[1], max_len=W, stride=STRIDE, text_bytes=len(q[0]), pair_bytes=len(ctx[0]),
                                  return_offsets_mapping=True)
    torch.cuda.synchronize()
    K = int(w["input_ids"].shape[0])
    by, ch = answers_for(ctx_strs, 5)
    d_by, d_ch = torch.from_numpy(by).to(dev), torch.from_numpy(ch).to(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    S = torch.randn((K, W), generator=g, device=dev)
    E = torch.randn((K, W), generator=g, device=dev)
    calls = {"qa_labels_bytes": lambda: tok.qa_labels(w, d_by),
             "qa_labels_chars": lambda: tok.qa_labels(w, d_ch, unit="char", context=dc),
             "qa_best_spans": lambda: tok.qa_best_spans(w, S, E, max_answer_len=L_)}
    res = {"workload": name, "docs": n, "max_len": W, "stride": STRIDE, "windows": K, "context_bytes": int(ctx[1][-1]), "max_answer_len": L_,
           "calls": {}}
    st_b, en_b = tok.qa_labels(w, d_by)
    st_c, en_c = tok.qa_labels(w, d_ch, unit="char", context=dc)
    assert torch.equal(st_b, st_c) and torch.equal(en_b, en_c)
    res["labelled_windows"] = int((st_b > 0).sum().item())
    for k, fn in calls.items():
        fn()
        ms = timed(fn, 20)
        tok.set_profiling(True); tok.profile_report(reset=True)
        fn(); torch.cuda.synchronize()
        prof = tok.profile_report(reset=True); tok.set_profiling(False)
        kern = {}
        for kn, v in prof.items():
            kern[kn] = {"launches": v["launches"], "ms": round(v["ms"], 4), "alg_bytes": v["alg_bytes"],
                        "alg_gb_per_s": v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] else None,
                        "share_of_measured_hbm": v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9 / bw if v["ms"] else None}
        res["calls"][k] = {"call_ms_median": float(np.median(ms)), "call_ms_best": min(ms), "kernels": kern}
    assert tok.check_errors(dev) == 0
    # host-side baselines on the same windows (numpy, a subset of the windows, scaled to all of them)
    om = w["offset_mapping"].cpu().numpy(); tt = w["token_type_ids"].cpu().numpy(); doc = w["overflow_to_sample_mapping"].cpu().numpy()
    rows = np.arange(0, K, max(1, K // 4000))
    t0 = time.perf_counter(); ns, ne = numpy_labels(om, tt, doc, by, rows); t1 = time.perf_counter()
    assert np.array_equal(ns, st_b.cpu().numpy()[rows]) and np.array_equal(ne, en_b.cpu().numpy()[rows])
    Sh, Eh = S.cpu().numpy(), E.cpu().numpy()
    t2 = time.perf_counter(); numpy_spans(Sh, Eh, om, tt, rows); t3 = time.perf_counter()
    t4 = time.perf_counter()
    conv = [(len(t[:a].encode("utf-8", "surrogatepass")), len(t[:b].encode("utf-8", "surrogatepass"))) for t, (a, b) in zip(ctx_strs, ch.tolist())]
    t5 = time.perf_counter()
    assert np.array_equal(np.array(conv), by)
    scale = K / len(rows)
    res["host_baselines"] = {"windows_timed": int(len(rows)),
                             "numpy_labels_ms_all_windows": (t1 - t0) * 1e3 * scale,
                             "numpy_best_span_search_ms_all_windows": (t3 - t2) * 1e3 * scale,
                             "python_char_to_byte_ms": (t5 - t4) * 1e3,
                             "note": "numpy per-window loops timed on every %d-th window and scaled to all windows; no cross-window reduction "
                                     "in the span search; the char conversion is len(ctx[:c].encode()) for both ends of every answer" % max(1, K // 4000)}
    print(json.dumps({"workload": name, "windows": K, "calls": {k: v["call_ms_median"] for k, v in res["calls"].items()},
                      "host": res["host_baselines"]}, default=float), flush=True)
    del w, S, E
    torch.cuda.empty_cache()
    return res


info = gpu_info()
bw = hbm_copy_gbs()
print(info, "measured HBM copy bandwidth %.0f GB/s" % bw, flush=True)
words = workload.default_wordlist().words
tok = Tokenize(devices=[0])
tok.set_option("max_chunk_bytes", 1 << 29)                   # one device call per workload (32,768 pairs: about 305 MB of context)
results = {"gpu": info, "hbm_copy_gb_per_s": bw, "cases": []}
for n in (4096, 32768):
    q = workload.generate(77, n, 5, 20, 0.0)
    ctx = workload.long_documents(words, n, lo=300, hi=1500, seed=9)
    results["cases"].append(case("%d question + context pairs" % n, tok, q, ctx, bw))
with open(os.path.join(out_dir, "qa_case.json"), "w") as f:
    json.dump(results, f, indent=1, default=float)
