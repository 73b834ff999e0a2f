"""Pair truncation strategies on one GPU: the stream path (k_rows<COUNT/RAGGED> per side -> k_pair_rows) against the reference cut
(truncation=True, the byte-parallel pipeline) on the same batch, device form (warm median, per-kernel split) and host form.
    python tools/truncation_case.py OUT_DIR        -> OUT_DIR/truncation_case.json
Workloads, 1,048,576 pairs each, produced on the device by workload.generate_hashed's generator (tok.synth_device):
  overflowing  NLI-like pairs (premise 20-300 words, hypothesis 3-20, 1 % noise words) at max_len 128: most premises do not fit,
               so longest_first cuts them and keeps the hypothesis.  About 1.1 GB of premises: the device form runs as four calls
               of 262,144 pairs (a device call holds at most max_chunk_bytes = 512 MiB), timed together.
  fit          the bench.py workload chunk (seed 1234, 3-13 words per side, no noise) at max_len 256: no row overflows, so every
               strategy gives the truncation=True row (checked here on every plane) and the difference is the price of the
               stream path against the byte-parallel pipeline.
"""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from genz_tokenize_b200 import Tokenize

out_dir = sys.argv[1]
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda:0")
N = 1 << 20


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"nvidia_smi": q.stdout.strip(), "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, reps):
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); r = fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms, r


def case(name, tok, parts, W, compare):
    """parts: [(side A, side B)] of (uint8 bytes tensor, int64 offsets tensor, byte count) on the device."""
    host = [tuple((t.cpu().numpy()[:nb], o.cpu().numpy()) for t, o, nb in pr) for pr in parts]
    def cat(side):                                                        # the whole batch on the host, offsets made absolute
        bs, offs, base = [], [np.zeros(1, dtype=np.int64)], 0
        for pr in host:
            bs.append(pr[side][0]); offs.append(pr[side][1][1:] + base); base += len(pr[side][0])
        return np.concatenate(bs), np.concatenate(offs)
    a, b = cat(0), cat(1)
    res = {"workload": name, "pairs": len(a[1]) - 1, "text_bytes": len(a[0]) + len(b[0]), "max_len": W, "device_calls": len(parts)}
    outs = {}
    for trunc in (True, "longest_first"):
        call = lambda: [tok.encode_device(A[0], A[1], B[0], B[1], max_len=W, sequence_id=False, text_bytes=A[2], pair_bytes=B[2], truncation=trunc)
                        for A, B in parts]
        call(); call()
        warm, r = timed(call, 7)
        assert tok.check_errors(dev) == 0
        tok.set_profiling(True); tok.profile_report(reset=True)
        call(); torch.cuda.synchronize()
        prof = tok.profile_report(reset=True); tok.set_profiling(False)
        r = {k: torch.cat([x[k] for x in r]) for k in r[0]}
        real = int(r["attention_mask"].sum().item())
        st = r["row_status"].cpu().numpy()
        key = "true" if trunc is True else trunc
        res[key] = {"device_warm_ms": warm, "device_warm_ms_median": float(np.median(warm)), "real_tokens": real,
                    "rows_at_max_len": int((r["row_len"] == W).sum().item()), "row_status_counts": np.bincount(st, minlength=3).tolist(),
                    "kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 4)} for k, v in prof.items()}}
        if compare:
            outs[key] = {k: v.cpu().numpy() for k, v in r.items()}
        del r
        tok.encode_batch(a, b, max_len=W, sequence_id=False, truncation=trunc)
        t0 = time.perf_counter(); hb = tok.encode_batch(a, b, max_len=W, sequence_id=False, truncation=trunc); t1 = time.perf_counter()
        res[key]["host_ms"] = (t1 - t0) * 1e3
        res[key]["host_d2h_bytes"] = hb.d2h_bytes
        del hb
        torch.cuda.empty_cache()
        print(name, key, json.dumps({k: res[key][k] for k in ("device_warm_ms_median", "host_ms", "row_status_counts")}), flush=True)
        print("  kernels:", {k: v["ms"] for k, v in res[key]["kernels"].items() if v["ms"] > 0.05}, flush=True)
    if compare:
        res["outputs_equal"] = all(np.array_equal(outs["true"][k], outs["longest_first"][k]) for k in outs["true"])
        assert res["outputs_equal"], "fit case: longest_first differs from truncation=True"
    res["longest_first_over_true_device"] = res["longest_first"]["device_warm_ms_median"] / res["true"]["device_warm_ms_median"]
    res["longest_first_over_true_host"] = res["longest_first"]["host_ms"] / res["true"]["host_ms"]
    return res


info = gpu_info()
print(info, flush=True)
tok = Tokenize(devices=[0])
tok.set_option("max_chunk_bytes", 1 << 29)                                   # the largest device call
results = {"gpu": info, "cases": []}
P = N // 4
nli = [(tok.synth_device(31, d0, P, 0, 20, 300, 0.01, device=dev), tok.synth_device(31, d0, P, 1, 3, 20, 0.01, device=dev)) for d0 in range(0, N, P)]
results["cases"].append(case("NLI-like overflowing pairs", tok, nli, 128, False))
del nli
torch.cuda.empty_cache()
fit = [(tok.synth_device(1234, 0, N, 0, 3, 13, 0.0, device=dev), tok.synth_device(1234, 0, N, 1, 3, 13, 0.0, device=dev))]
results["cases"].append(case("bench.py chunk (every row fits)", tok, fit, 256, True))
with open(os.path.join(out_dir, "truncation_case.json"), "w") as f:
    json.dump(results, f, indent=1, default=float)
