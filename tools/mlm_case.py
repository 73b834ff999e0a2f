"""Masked-language-model masking on one GPU: Tokenize.mlm_mask (token and whole-word) on two id planes of the sizes pre-training
runs, against a device-to-device copy of the same byte count and against HF's recipe restated in torch ops, all in one run.
    python tools/mlm_case.py OUT_DIR        -> OUT_DIR/mlm_case.json
Workloads: 1,048,576 synthetic single sentences of 20-100 words (workload.generate_hashed made on the device by synth_device) at
max_len=128 through encode_device, and windows of long documents (6,000-9,000 words, workload.long_documents) at max_len=512 /
stride=128 through encode_windows_device, at least 262,144 windows.  Every plane is far larger than the 126 MB L2 (the 128-column
plane reads 512 MiB and writes 1.5 GiB per call), so each call streams from HBM.
Per workload and mode: the kernel's time from the library's CUDA events (set_profiling) over >= 0.5 s of calls after a warm-up, its
bytes per second from 16 B per column (4 read, 4 + 8 written), and the same from a torch device-to-device copy of 8 B per column
(8 read + 8 written, the same 16 B per column) timed in the same run; the call time of the Python method; and, token mode only,
HF's DataCollatorForLanguageModeling recipe restated in torch ops on the same plane (torch cannot group BPE pieces into words)."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from genz_tokenize_b200 import Tokenize, workload

out_dir = sys.argv[1]
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda:0")
MIN_S = 0.5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"nvidia_smi": q.stdout.strip(), "torch_name": torch.cuda.get_device_name(0)}


def timed_loop(fn):
    """(ms per call, calls): event-timed loops of doubling length until one lasts >= MIN_S."""
    fn(); fn()
    torch.cuda.synchronize()
    reps = 4
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= MIN_S * 1e3:
            return ms / reps, reps
        reps *= 2


def hf_torch(ids, special, mask_id, n_vocab, gen, p=0.15):
    """DataCollatorForLanguageModeling.torch_mask_tokens (transformers 4.x), token mode, in torch ops."""
    labels = ids.long()
    prob = torch.full(labels.shape, p, device=ids.device)
    prob.masked_fill_(torch.isin(ids, special), 0.0)
    masked = torch.bernoulli(prob, generator=gen).bool()
    labels = torch.where(masked, labels, -100)
    replaced = torch.bernoulli(torch.full(labels.shape, 0.8, device=ids.device), generator=gen).bool() & masked
    inputs = torch.where(replaced, mask_id, ids)
    rnd = torch.bernoulli(torch.full(labels.shape, 0.5, device=ids.device), generator=gen).bool() & masked & ~replaced
    words = torch.randint(n_vocab, labels.shape, dtype=torch.int32, device=ids.device, generator=gen)
    inputs = torch.where(rnd, words, inputs)
    return inputs, labels


def case(name, tok, ids, bw_copy):
    n, W = ids.shape
    cols = n * W
    sp = torch.tensor(tok._special_ids(), dtype=torch.int32, device=dev)
    res = {"workload": name, "rows": n, "max_len": W, "columns": cols, "alg_bytes_per_call": 16 * cols,
           "real_tokens": int(((ids >= 0) & ~torch.isin(ids, sp)).sum()), "modes": {}}
    for ww in (False, True):
        mode = "whole_word" if ww else "token"
        call = lambda: tok.mlm_mask(ids, 1234, whole_word=ww)
        _, lab = call()
        res["modes"][mode] = {"selected_fraction_of_eligible": float((lab != -100).sum()) / res["real_tokens"]}
        del lab
        call_ms, reps = timed_loop(call)
        tok.set_profiling(True); tok.profile_report(reset=True)
        t0 = time.perf_counter()
        k = 0
        while time.perf_counter() - t0 < MIN_S or k < 8:
            call(); k += 1
        torch.cuda.synchronize()
        prof = tok.profile_report(reset=True); tok.set_profiling(False)
        kn = "k_mlm_mask_words" if ww else "k_mlm_mask_tokens"
        kms = prof[kn]["ms"] / prof[kn]["launches"]
        gbs = 16 * cols / (kms * 1e-3) / 1e9
        res["modes"][mode].update({"kernel": kn, "kernel_launches_timed": prof[kn]["launches"], "kernel_ms": kms, "kernel_gb_per_s": gbs,
                                   "share_of_measured_copy": gbs / bw_copy(cols), "call_ms": call_ms, "calls_timed": reps,
                                   "launches_per_call": prof[kn]["launches"] / k})
    # the same recipe in torch ops, on the same plane
    gen = torch.Generator(device=dev).manual_seed(0)
    n_vocab = tok.vocab_size()
    msk = tok._special_ids()[3]
    hf_ms, reps = timed_loop(lambda: hf_torch(ids, sp, msk, n_vocab, gen))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        hf_torch(ids, sp, msk, n_vocab, gen)
        torch.cuda.synchronize()
    kernels = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
    res["hf_recipe_torch_ops"] = {"ms": hf_ms, "calls_timed": reps, "cuda_kernels_per_call": kernels,
                                  "speedup_of_token_mode_call": hf_ms / res["modes"]["token"]["call_ms"]}
    print(json.dumps({"workload": name, "rows": n, "W": W,
                      "kernel_ms_and_share_of_copy": {m: (v["kernel_ms"], v["share_of_measured_copy"]) for m, v in res["modes"].items()},
                      "hf_torch_ms": hf_ms}), flush=True)
    return res


copy_cache = {}


def copy_gbs(cols):
    """Measured device-to-device copy of a buffer of 8 B per column: (read + write) bytes per second, in the same run."""
    if cols not in copy_cache:
        a = torch.empty((cols * 8,), dtype=torch.uint8, device=dev)
        b = torch.empty_like(a)
        ms, _ = timed_loop(lambda: b.copy_(a))
        copy_cache[cols] = 16 * cols / (ms * 1e-3) / 1e9
        del a, b
        torch.cuda.empty_cache()
    return copy_cache[cols]


info = gpu_info()
print(info, flush=True)
tok = Tokenize(devices=[0])
tok.set_option("max_chunk_bytes", 1 << 29)                   # a batch of 1,000 long documents is about 75 MiB of text: one device call
results = {"gpu": info, "cases": []}

# 1. 1,048,576 synthetic singles at max_len=128, encoded in pieces (a device call takes at most max_chunk_bytes of text)
N1, PIECE = 1 << 20, 1 << 16
planes = []
for d0 in range(0, N1, PIECE):
    data, off, nb = tok.synth_device(7, d0, PIECE, lo=20, hi=100, device=dev)
    planes.append(tok.encode_device(data, off, max_len=128, text_bytes=nb)["input_ids"])
ids = torch.cat(planes)
del planes, data, off
torch.cuda.synchronize(); torch.cuda.empty_cache()
results["cases"].append(case("1,048,576 synthetic singles, 20-100 words, max_len=128", tok, ids, copy_gbs))
del ids
torch.cuda.empty_cache()

# 2. windows of long documents at max_len=512, stride=128
words = workload.default_wordlist().words
planes, K, seed = [], 0, 0
while K < 262144:
    b, o = workload.long_documents(words, 1000, seed=100 + seed)
    up = torch.from_numpy(np.concatenate([b, np.zeros((-len(b)) % 16 + 32, dtype=np.uint8)])).to(dev)
    w = tok.encode_windows_device(up, torch.from_numpy(o).to(dev), max_len=512, stride=128, text_bytes=len(b))
    planes.append(w["input_ids"])
    K += int(w["input_ids"].shape[0])
    seed += 1
ids = torch.cat(planes)
del planes, w, up
torch.cuda.synchronize(); torch.cuda.empty_cache()
results["cases"].append(case("%d windows of %d long documents (6,000-9,000 words), max_len=512, stride=128" % (K, 1000 * seed), tok, ids, copy_gbs))
assert tok.check_errors(dev) == 0
with open(os.path.join(out_dir, "mlm_case.json"), "w") as f:
    json.dump(results, f, indent=1, default=float)
