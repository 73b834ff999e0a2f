"""Long documents as windows on one GPU: device form (cold / warm call time, per-kernel split), host form end to end, and the
fixed-layout encode of the same documents (first window only) as the reference point.
    python tools/windows_case.py OUT_DIR        -> OUT_DIR/windows_case.json
Workloads: 4,096 long documents (bundled word list, 6,000-9,000 words) at max_len=512 / stride=128 and at max_len=4096 / stride=0;
4,096 question + context pairs (5-20 word questions, 300-1,500 word contexts) at max_len=384 / stride=128.  The text is far larger
than the 126 MB L2; the token streams of one call are about its size, and the planes being written push them out."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from genz_tokenize_b200 import Tokenize, workload

out_dir = sys.argv[1]
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda:0")


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


def up(a):
    return torch.from_numpy(np.concatenate([a, np.zeros((-len(a)) % 16 + 32, dtype=np.uint8)])).to(dev)


def timed(fn, reps):
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); r = fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms, r


def case(name, tok, a, b, W, s, bw):
    n = len(a[1]) - 1
    text_bytes = int(a[1][-1]) + (int(b[1][-1]) if b is not None else 0)
    da = (up(a[0]), torch.from_numpy(a[1]).to(dev), len(a[0]))
    db = (up(b[0]), torch.from_numpy(b[1]).to(dev), len(b[0])) if b is not None else (None, None, None)
    call = lambda: tok.encode_windows_device(da[0], da[1], db[0], db[1], max_len=W, stride=s, text_bytes=da[2], pair_bytes=db[2])
    call()
    tok.cache_reset()
    cold, _ = timed(call, 1)
    warm, r = timed(call, 10)
    assert tok.check_errors(dev) == 0
    K = int(r["input_ids"].shape[0])
    real = int(r["attention_mask"].sum().item())
    # per-kernel split, in a run of its own
    tok.set_profiling(True); tok.profile_report(reset=True)
    call(); torch.cuda.synchronize()
    prof = tok.profile_report(reset=True); tok.set_profiling(False)
    planes_b = K * W * (5 + (1 if b is not None else 0))
    maps_b = K * (8 + 4 + 4 + (5 if b is not None else 0)) + (n + 1) * 8
    alg = text_bytes + 8 * (n + 1) * (2 if b is not None else 1) + planes_b + maps_b
    wr = prof.get("k_window_rows", {})
    # what k_window_rows reads besides: every window's tokens from the token streams (4 bytes per real token that is not
    # framing; the streams of these workloads are larger than L2, so most of it comes from HBM)
    reads = 4 * (real - K * (4 if b is not None else 2))
    warm_ms = float(np.median(warm))
    res = {"workload": name, "docs": n, "text_bytes": text_bytes, "max_len": W, "stride": s, "windows": K, "real_tokens": real,
           "device_form": {"cold_ms": cold[0], "warm_ms": warm, "warm_ms_median": warm_ms, "warm_ms_best": min(warm), "windows_per_s": K / (warm_ms * 1e-3),
                           "real_tokens_per_s": real / (warm_ms * 1e-3), "alg_bytes": alg, "alg_gb_per_s": alg / (warm_ms * 1e-3) / 1e9,
                           "share_of_measured_hbm": alg / (warm_ms * 1e-3) / 1e9 / bw},
           "kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 4), "alg_bytes": v["alg_bytes"]} for k, v in prof.items()},
           "k_window_rows": {"ms": wr.get("ms"), "alg_bytes": wr.get("alg_bytes"),
                             "alg_gb_per_s": wr["alg_bytes"] / (wr["ms"] * 1e-3) / 1e9 if wr.get("ms") else None,
                             "share_of_measured_hbm": wr["alg_bytes"] / (wr["ms"] * 1e-3) / 1e9 / bw if wr.get("ms") else None,
                             "stream_read_bytes": reads,
                             "share_of_measured_hbm_with_stream_reads": (wr["alg_bytes"] + reads) / (wr["ms"] * 1e-3) / 1e9 / bw if wr.get("ms") else None}}
    del r
    # host form, end to end (host arrays in, pinned host planes out)
    tok.encode_windows(a, b, max_len=W, stride=s)
    t0 = time.perf_counter(); hw = tok.encode_windows(a, b, max_len=W, stride=s); t1 = time.perf_counter()
    assert len(hw["input_ids"]) == K
    del hw
    res["host_form_ms"] = (t1 - t0) * 1e3
    # the fixed-layout encode of the same documents: the first window of each only
    call_fixed = lambda: tok.encode_device(da[0], da[1], db[0], db[1], max_len=W, text_bytes=da[2], pair_bytes=db[2])
    call_fixed()
    fx, _ = timed(call_fixed, 5)
    tok.encode_batch(a, b, max_len=W)
    t0 = time.perf_counter(); tok.encode_batch(a, b, max_len=W); t1 = time.perf_counter()
    res["first_window_only"] = {"device_warm_ms_median": float(np.median(fx)), "host_ms": (t1 - t0) * 1e3}
    torch.cuda.empty_cache()
    print(json.dumps({k: res[k] for k in ("workload", "windows", "device_form", "host_form_ms")}, default=float), flush=True)
    print("  kernels:", {k: v["ms"] for k, v in res["kernels"].items() if v["ms"] > 0.05}, flush=True)
    return res


info = gpu_info()
bw = hbm_copy_gbs()
print(info, "measured HBM copy bandwidth %.0f GB/s" % bw, flush=True)
words = workload.default_wordlist().words
docs = workload.long_documents(words, 4096)
q = workload.generate(77, 4096, 5, 20, 0.0)
ctx = workload.long_documents(words, 4096, lo=300, hi=1500, seed=9)
tok = Tokenize(devices=[0])
tok.set_option("max_chunk_bytes", 1 << int(np.ceil(np.log2(len(docs[0]) + (1 << 20)))))     # one device call per workload
results = {"gpu": info, "hbm_copy_gb_per_s": bw, "cases": []}
for name, a, b, W, s in (("4096 long documents", docs, None, 512, 128), ("4096 long documents", docs, None, 4096, 0),
                         ("4096 question + context pairs", q, ctx, 384, 128)):
    results["cases"].append(case(name, tok, a, b, W, s, bw))
with open(os.path.join(out_dir, "windows_case.json"), "w") as f:
    json.dump(results, f, indent=1, default=float)
