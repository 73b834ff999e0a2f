"""BPE-dropout on one GPU: encode_device(..., bpe_dropout=p) at p = 0 and p = 0.1 against encode_device on a warm word cache, on the
same batch, device form (CUDA events around the call, median of 5 after 2 warm-up calls, per-kernel split from a profiled call).
    python tools/dropout_case.py OUT_DIR        -> OUT_DIR/dropout_case.json
Workloads, produced on the device by workload.generate_hashed's generator (tok.synth_device):
  pairs    the bench.py workload chunk: 1,048,576 pairs, seed 1234, 3-13 words per side, no noise, max_len 256
  singles  1,048,576 single sentences of 3-40 words, 1 % noise words, max_len 128
  long     32,768 documents of 300-2,000 words, 1 % noise words, max_len 512: the dropout walk stops once a text has 512 ids
The p = 0 rows are checked against the encode_device rows on every plane.  Rates are real tokens (attention_mask ones) per second.
"""
import json, os, subprocess, sys
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


def case(name, tok, A, B, W):
    res = {"workload": name, "docs": A[1].numel() - 1, "text_bytes": A[2] + (B[2] if B else 0), "max_len": W}
    outs = {}
    for key, p in (("encode_device_warm", None), ("dropout_p0", 0.0), ("dropout_p0.1", 0.1)):
        call = lambda: tok.encode_device(A[0], A[1], B[0] if B else None, B[1] if B else None, max_len=W, sequence_id=True, text_bytes=A[2],
                                         pair_bytes=B[2] if B else None, bpe_dropout=p, seed=1)
        call(); call()
        ms, r = timed(call, 5)
        assert tok.check_errors(dev) == 0
        tok.set_profiling(True); tok.profile_report(reset=True)
        call(); torch.cuda.synchronize()
        prof = tok.profile_report(reset=True); tok.set_profiling(False)
        real = int(r["attention_mask"].sum().item())
        med = float(np.median(ms))
        res[key] = {"device_ms": ms, "device_ms_median": med, "real_tokens": real, "tokens_per_s": real / med * 1e3,
                    "kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 4)} for k, v in prof.items()}}
        if p != 0.1:
            outs[key] = {k: v.cpu().numpy() for k, v in r.items()}
        del r
        print(name, key, json.dumps({k: res[key][k] for k in ("device_ms_median", "tokens_per_s")}), flush=True)
        print("  kernels:", {k: v["ms"] for k, v in res[key]["kernels"].items() if v["ms"] > 0.05}, flush=True)
    res["p0_equals_encode_device"] = all(np.array_equal(outs["dropout_p0"][k], outs["encode_device_warm"][k]) for k in outs["dropout_p0"])
    assert res["p0_equals_encode_device"], name
    for key in ("dropout_p0", "dropout_p0.1"):
        res[key + "_over_encode_device"] = res[key]["device_ms_median"] / res["encode_device_warm"]["device_ms_median"]
    return res


info = gpu_info()
print(info, flush=True)
tok = Tokenize(devices=[0])
tok.set_option("max_chunk_bytes", 1 << 29)                                   # the largest device call
results = {"gpu": info, "cases": []}
for name, W, A, B in (("bench.py pairs", 256, (1234, N, 0, 3, 13, 0.0), (1234, N, 1, 3, 13, 0.0)),
                      ("singles", 128, (77, N, 0, 3, 40, 0.01), None),
                      ("long documents", 512, (55, N // 32, 0, 300, 2000, 0.01), None)):
    synth = lambda s: tok.synth_device(s[0], 0, s[1], s[2], s[3], s[4], s[5], device=dev)
    results["cases"].append(case(name, tok, synth(A), synth(B) if B else None, W))
    torch.cuda.empty_cache()
with open(os.path.join(out_dir, "dropout_case.json"), "w") as f:
    json.dump(results, f, indent=1, default=float)
