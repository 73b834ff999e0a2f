"""offset_mapping on one GPU: what asking for token offsets costs.
    python tools/offsets_case.py OUT_DIR        -> OUT_DIR/offsets_case.json
Workloads: the three of tools/windows_case.py through the device form (encode_windows_device), with and without offsets -- cold
and warm call time, the per-kernel split and k_window_rows' bytes against the measured HBM copy bandwidth -- and the reference's
default call shape (1,048,576 single sentences, max_len None: ragged) through the host API as tools/ragged_case.py runs it."""
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


def windows_case(name, tok, a, b, W, s, bw):
    da = (up(a[0]), torch.from_numpy(a[1]).to(dev), len(a[0]))
    db = (up(b[0]), torch.from_numpy(b[1]).to(dev), len(b[0])) if b is not None else (None, None, None)
    res = {"workload": name, "docs": len(a[1]) - 1, "max_len": W, "stride": s}
    for offs in (False, True):
        call = lambda: tok.encode_windows_device(da[0], da[1], db[0], db[1], max_len=W, stride=s, text_bytes=da[2], pair_bytes=db[2],
                                                 return_offsets_mapping=offs)
        call()
        tok.cache_reset()
        cold, _ = timed(call, 1)
        warm, r = timed(call, 10)
        assert tok.check_errors(dev) == 0
        K = int(r["input_ids"].shape[0])
        del r
        tok.set_profiling(True); tok.profile_report(reset=True)
        call(); torch.cuda.synchronize()
        prof = tok.profile_report(reset=True); tok.set_profiling(False)
        wr = prof.get("k_window_rows_offsets" if offs else "k_window_rows", {})
        warm_ms = float(np.median(warm))
        res["offsets" if offs else "plain"] = {
            "windows": K, "cold_ms": cold[0], "warm_ms": warm, "warm_ms_median": warm_ms, "windows_per_s": K / (warm_ms * 1e-3),
            "kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 4), "alg_bytes": v["alg_bytes"]} for k, v in prof.items()},
            "k_window_rows": {"ms": wr.get("ms"), "alg_bytes": wr.get("alg_bytes"),
                              "alg_gb_per_s": wr["alg_bytes"] / (wr["ms"] * 1e-3) / 1e9 if wr.get("ms") else None,
                              "share_of_measured_hbm": wr["alg_bytes"] / (wr["ms"] * 1e-3) / 1e9 / bw if wr.get("ms") else None}}
        torch.cuda.empty_cache()
    res["warm_ratio"] = res["offsets"]["warm_ms_median"] / res["plain"]["warm_ms_median"]
    print(json.dumps({"workload": name, "W": W, "plain_ms": res["plain"]["warm_ms_median"], "offsets_ms": res["offsets"]["warm_ms_median"],
                      "k_window_rows": [res[k]["k_window_rows"]["ms"] for k in ("plain", "offsets")]}), flush=True)
    return res


def ragged_case(tok):
    n = 1 << 20
    tb, to = workload.generate(1234, n, 3, 13, 0.0)
    res = {"workload": "1,048,576 single sentences, max_len None (ragged), host API, pageable text", "docs": n, "text_bytes": len(tb)}
    for offs in (False, True):
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            be = tok.encode_batch((tb, to), return_offsets_mapping=offs)
            ts.append((time.perf_counter() - t0) * 1e3)
            toks = int(be["real_tokens"]); d2h = be.d2h_bytes
            del be
        tok.set_profiling(True); tok.profile_report(reset=True)
        be = tok.encode_batch((tb, to), return_offsets_mapping=offs); del be
        prof = tok.profile_report(reset=True); tok.set_profiling(False)
        res["offsets" if offs else "plain"] = {"ms_per_call": ts, "best_ms": min(ts[1:]), "real_tokens": toks, "d2h_bytes": d2h,
                                               "kernel_ms": sum(v["ms"] for v in prof.values()),
                                               "kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 4)} for k, v in prof.items()}}
    print(json.dumps({"workload": res["workload"], "plain_best_ms": res["plain"]["best_ms"], "offsets_best_ms": res["offsets"]["best_ms"],
                      "kernel_ms": [res[k]["kernel_ms"] for k in ("plain", "offsets")]}), flush=True)
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
results = {"gpu": info, "hbm_copy_gb_per_s": bw, "windows": [], "ragged": None}
for name, a, b, W, s in (("4096 long documents", docs, None, 512, 128), ("4096 long documents", docs, None, 4096, 0),
                         ("4096 question + context pairs", q, ctx, 384, 128)):
    results["windows"].append(windows_case(name, tok, a, b, W, s, bw))
results["ragged"] = ragged_case(Tokenize(devices=[0]))
with open(os.path.join(out_dir, "offsets_case.json"), "w") as f:                # one line per workload
    f.write("{\n" + ",\n".join(json.dumps(k) + ": " + json.dumps(v, default=float) for k, v in results.items() if k != "windows"))
    f.write(',\n"windows": [\n' + ",\n".join(json.dumps(c, default=float) for c in results["windows"]) + "\n]\n}\n")
