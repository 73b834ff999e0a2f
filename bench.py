#!/usr/bin/env python3
"""bench.py -- the encode hot path on N B200s (one process per GPU) on BASELINE.json configs[2], next to the reference.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--pairs P] [--chunk C]

Workload (BASELINE configs[2]): bundled vocab, P = 100,000,000 synthetic sentence pairs (3-13 words a side sampled from
vocab.txt in proportion to the counts, ~101 B of UTF-8 per pair, SURVEY.md 8 d2), max_len=256, padding + truncation, three
planes (input_ids int32, attention_mask uint8, token_type_ids int8).  The batch shards by document: rank r owns pairs
[P r / N, P (r + 1) / N) -- STRONG scaling, no collective on the data path (NCCL carries the barrier and the timing only).
A rank's share is produced on its GPU by the counter-based generator (workload.generate_hashed / csrc/synth.cuh, untimed),
stays resident in HBM, and is streamed through the CUDA pipeline in chunks of C = 1,048,576 pairs into ONE reused set of
[C, 256] output planes (165 GB of planes do not fit beside the text).  One step = one pass over the rank's whole share.

Prints ONE JSON line (rank 0):
  value        real tokens/s, whole job, text resident in HBM, planes written to HBM (CUDA events around every pass, max over ranks)
  roofline     the dominant kernel: algorithmic bytes per launch / its CUDA-event duration against the measured HBM copy bandwidth;
               roofline.whole_path = SURVEY.md 8 d4 bytes of a step / step time (the number to hold against the 50 % target)
  digest       order-independent 64-bit digest of all output planes of the batch: equal at N = 1, 2, 4, 8 (SURVEY.md 8 d7)
  cold / noise the first pass after a cache reset, and a pass over text with 1 % adversarial words (fresh words every chunk: the
               BPE kernel k_bpe_pending works in steady state)
  e2e          the same metric through Tokenize.encode_batch with HOST buffers (pinned text in, pinned planes out), copies timed
  cpu_baseline the UNMODIFIED Python reference (oracle/_ref) on this host: one process and multiprocessing.Pool(all cores); the C
               restatement (oracle/) beside it
  extra        BASELINE configs[1] (1M singles, max_len 128: device-resident, cold, and end to end through the host API), configs[3] (decode of
               the planes into a reused text ring), the reference's default call shape (ragged rows, host API), configs[4] (custom vocab,
               long documents, cold and warm)
`--impl reference` times the reference itself (Pool over all cores) on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step left in the output planes (its last chunk) as DIR/<plane>.npy, float32:
a fixed, seeded sample of DUMP_ROWS rows, with their global pair indices in DIR/pair_index.npy (float64), so that two builds
can be compared output for output on the same arguments.
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAIRS = 100_000_000
CHUNK = 1 << 20
MAX_LEN = 256
SEED = 1234
LO, HI = 3, 13
NOMINAL_HBM_GBS = 8000.0          # north_star's figure; the measured copy bandwidth is the other denominator (SURVEY.md 8 d3)
REF_SAMPLE_PAIRS = 40960           # --impl reference: pairs per step (the first pairs of the global batch)
L2_FLUSH_BYTES = 256 << 20
DUMP_ROWS = 16384                  # --dump-outputs: 16,384 rows x 256 x 3 planes x 4 B = 48 MiB of float32, under 64 MB in all
DUMP_SEED = 20240601


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def workload_name(pairs):
    return ("bundled vocab, %d synthetic sentence pairs (3-13 words a side, ~101 B UTF-8 per pair), max_len=256, padding+truncation, "
            "input_ids+attention_mask+token_type_ids (BASELINE configs[2])" % pairs)


def source_hash():
    """Hash of the CUDA sources: ties profiles/roofline_traffic.json to the build it was captured on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "genz_tokenize_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".hpp")):
            with open(os.path.join(d, f), "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()[:16]


class ClockSampler:
    """Samples SM clock + throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.max_mhz = [], set(), False, None
        self.busy = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        nv = self.nv
        names = {"hw_slowdown": "nvmlClocksEventReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksEventReasonHwThermalSlowdown",
                 "sw_thermal_slowdown": "nvmlClocksEventReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksEventReasonSwPowerCap"}
        alt = {"hw_slowdown": "nvmlClocksThrottleReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksThrottleReasonHwThermalSlowdown",
               "sw_thermal_slowdown": "nvmlClocksThrottleReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksThrottleReasonSwPowerCap"}
        while not self.stop_flag:
            try:
                if self.busy:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for k in names:
                        bit = getattr(nv, names[k], None) or getattr(nv, alt[k], 0)
                        if r & bit:
                            self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self.t.start()

    def stop(self):
        self.stop_flag = True
        if self.nv and self.t.is_alive():
            self.t.join(timeout=1)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------------------------------------------------
def host_pairs(n, doc0=0, noise=0.0):
    """The first n pairs of the global batch on the host: (packed A, packed B, list[str] A, list[str] B)."""
    from genz_tokenize_b200 import workload
    a = workload.generate_hashed(SEED, doc0, n, 0, LO, HI, noise)
    b = workload.generate_hashed(SEED, doc0, n, 1, LO, HI, noise)
    return a, b, workload.unpack(*a), workload.unpack(*b)


def port_rate(a, b, threads, repeats=1):
    """pairs/s and tokens/s of the C restatement (oracle/genztok_oracle.c) on packed pairs."""
    from oracle.oracle import Oracle
    o = Oracle()
    best, toks = None, 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = o.encode_batch(a, b, max_len=MAX_LEN, threads=threads)
        dt = time.perf_counter() - t0
        toks = int(r["mask"].sum())
        best = dt if best is None or dt < best else best
    return toks / best, toks, best


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_baseline_block():
    """The reference on this host's cores, same run (SURVEY.md 8 d6): Python single process + Pool(all cores); the C port beside it."""
    cores = host_threads()
    blk = {"unit": "tokens/s", "cores": cores, "cpu_model": cpu_model()}
    from oracle import ref_pool
    n_single, n_pool = 10240, max(204800, 4096 * cores)
    (a, b, ta, tb_) = host_pairs(n_pool)
    if ref_pool.available():
        toks, dt = ref_pool.encode_single(ta[:n_single], tb_[:n_single], MAX_LEN)
        blk["python_single"] = {"pairs": n_single, "seconds": dt, "pairs_per_s": n_single / dt, "tokens_per_s": toks / dt, "processes": 1}
        pool = ref_pool.RefPool(cores, 500)
        try:
            toks, dt = pool.encode(ta, tb_, MAX_LEN)
        finally:
            pool.close()
        blk["python_pool"] = {"pairs": n_pool, "seconds": dt, "pairs_per_s": n_pool / dt, "tokens_per_s": toks / dt, "processes": cores, "job_docs": 500}
        blk["value"], blk["kind"] = toks / dt, "reference"
        blk["sample"] = ("the UNMODIFIED reference (oracle/_ref = /root/reference/genz_tokenize/tokenize.py) on the first %d pairs of the batch with "
                         "multiprocessing.Pool(%d), 500-pair jobs, one Tokenize() per worker (%.1f s); one process on the first %d pairs (%.1f s)"
                         % (n_pool, cores, dt, n_single, blk["python_single"]["seconds"]))
    try:
        from oracle.oracle import Oracle
        threads = max(Oracle.max_threads(), cores)
        sub = lambda p, n: (p[0][:p[1][n]], p[1][:n + 1])
        r1, _, dt1 = port_rate(sub(a, 65536), sub(b, 65536), 1)
        rN, _, dtN = port_rate(a, b, threads, repeats=3)
        blk["port"] = {"kind": "port", "what": "oracle/genztok_oracle.c, the C restatement of tokenize.py (no memoisation), OpenMP over documents",
                       "threads": threads, "tokens_per_s": rN, "single_thread_tokens_per_s": r1, "pairs": n_pool, "seconds": dtN}
        if "value" not in blk:
            blk["value"], blk["kind"] = rN, "port"
            blk["sample"] = "oracle/_ref is absent: the C restatement on the first %d pairs with %d OpenMP threads (%.2f s)" % (n_pool, threads, dtN)
    except Exception as e:          # the baseline is reporting only; never fail the GPU line over it
        blk["port"] = {"failed": repr(e)}
    return blk


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path with all host cores, on a bounded sample per step."""
    if rank != 0:
        return
    from oracle import ref_pool
    cores = host_threads()
    n = REF_SAMPLE_PAIRS
    a, b, ta, tb_ = host_pairs(n)
    in_bytes = int(a[1][-1] + b[1][-1])
    use_ref = ref_pool.available()
    if use_ref:
        pool = ref_pool.RefPool(cores, 500)
        step = lambda: pool.encode(ta, tb_, MAX_LEN)
        kind, what = "reference", "the UNMODIFIED reference (oracle/_ref) in multiprocessing.Pool(%d), 500-pair jobs" % cores
    else:
        from oracle.oracle import Oracle
        threads = max(Oracle.max_threads(), cores)
        step = lambda: port_rate(a, b, threads)[1:]
        kind, what = "port", "oracle/_ref absent: oracle/genztok_oracle.c with %d OpenMP threads" % threads
    for _ in range(max(args.warmup, 0)):
        step()
    t_tot, tok_tot = 0.0, 0
    for _ in range(args.steps):
        toks, dt = step()
        t_tot += dt
        tok_tot += toks
    if use_ref:
        pool.close()
    value = tok_tot / t_tot
    line = {
        "impl": "reference", "metric": "encode_tokens_per_sec", "value": value, "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
        "config": {"workload": workload_name(args.pairs), "max_len": MAX_LEN,
                   "sample": "each step = the first %d pairs of the batch (the whole batch would take hours on the host); rates are per token, so they compare" % n},
        "pairs_per_s": n * args.steps / t_tot, "input_gb_per_s": in_bytes * args.steps / t_tot / 1e9,
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": cores, "kind": kind, "cpu_model": cpu_model(), "sample": "%s, %d pairs per step" % (what, n)},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
class Stream:
    """One rank's share of the batch resident in HBM + the reused output planes; encode(c) enqueues chunk c."""

    def __init__(self, tok, torch, dev, doc0, n, chunk, noise=0.0, seed=SEED, planes=None):
        self.tok, self.torch, self.dev, self.doc0, self.n, self.chunk = tok, torch, dev, doc0, n, chunk
        self.text, self.toff, self.tbytes = tok.synth_device(seed, doc0, n, 0, LO, HI, noise, device=dev)
        self.pair, self.poff, self.pbytes = tok.synth_device(seed, doc0, n, 1, LO, HI, noise, device=dev)
        self.starts = list(range(0, n, chunk))
        idx = torch.tensor(self.starts + [n], dtype=torch.int64, device=dev)
        self.tcut = self.toff[idx].cpu().tolist()
        self.pcut = self.poff[idx].cpu().tolist()
        m = min(chunk, n)
        if planes is None:
            planes = {"input_ids": torch.empty((m, MAX_LEN), dtype=torch.int32, device=dev), "attention_mask": torch.empty((m, MAX_LEN), dtype=torch.uint8, device=dev),
                      "token_type_ids": torch.empty((m, MAX_LEN), dtype=torch.int8, device=dev), "row_len": torch.empty((m,), dtype=torch.int32, device=dev),
                      "seq_len": torch.empty((m,), dtype=torch.int32, device=dev), "row_status": torch.empty((m,), dtype=torch.uint8, device=dev)}
        self.planes = planes
        self.calls = []
        for c, s in enumerate(self.starts):
            e = min(n, s + chunk)
            out = planes if e - s == m else {k: v[:e - s] for k, v in planes.items()}
            self.calls.append((self.toff[s:e + 1], self.poff[s:e + 1], out, self.tcut[c + 1] - self.tcut[c], self.pcut[c + 1] - self.pcut[c], s))
        self.in_bytes = self.tbytes + self.pbytes

    def encode(self, c):
        to, po, out, tb, pb, _ = self.calls[c]
        self.tok.encode_device(self.text, to, self.pair, po, max_len=MAX_LEN, out=out, text_bytes=tb, pair_bytes=pb)
        return out

    def run_pass(self, chunks=None):
        for c in (range(len(self.calls)) if chunks is None else chunks):
            self.encode(c)

    def alg_bytes(self, chunks=None):
        """SURVEY.md 8 d4: utf8 of both sides + 8 (n + 1) per side + n * 256 * (4 + 1 + 1)."""
        tot = 0
        for c in (range(len(self.calls)) if chunks is None else chunks):
            to, _, _, tb, pb, _ = self.calls[c]
            m = to.numel() - 1
            tot += tb + pb + 16 * (m + 1) + m * MAX_LEN * 6
        return tot


def dump_outputs(out, row0, path, max_rows=DUMP_ROWS):
    """A fixed, seeded sample of the rows of the planes `out` (rows row0 ... of the batch) -> path/<plane>.npy as float32 (every
    value is an integer below 2^24), and path/pair_index.npy (float64): the global pair index of each sampled row."""
    import torch
    m = out["input_ids"].shape[0]
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(m, size=min(m, max_rows), replace=False))
    idx = torch.from_numpy(rows).to(out["input_ids"].device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "pair_index.npy"), (row0 + rows).astype(np.float64))
    for name, plane in out.items():
        np.save(os.path.join(path, name + ".npy"), plane.index_select(0, idx).cpu().numpy().astype(np.float32))


def timed_passes(torch, fn, reps):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def kernel_table(prof, reps, peak):
    out = {}
    for name, v in prof.items():
        L = max(v["launches"], 1)
        ent = {"ms": v["ms"] / L, "launches": v["launches"] / reps}
        if v.get("alg_bytes"):
            ent["alg_bytes"] = v["alg_bytes"] / L
            ent["alg_gb_per_s"] = ent["alg_bytes"] / (ent["ms"] * 1e-3) / 1e9
            ent["frac_of_peak"] = ent["alg_gb_per_s"] / peak
        out[name] = ent
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=env_int("GENZTOK_BENCH_PAIRS", PAIRS), help="sentence pairs in the GLOBAL batch (default: BASELINE configs[2])")
    ap.add_argument("--chunk", type=int, default=CHUNK, help="pairs per pass through the reused output planes")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-pairs", type=int, default=2 * CHUNK, help="pairs per rank of the end-to-end (host buffers) leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip configs[1] / [3] / [4] side measurements")
    ap.add_argument("--no-arms", action="store_true", help="skip the cold / noise arms")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a sample of the planes of the last timed step to DIR/<plane>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    from genz_tokenize_b200 import Tokenize, workload
    from genz_tokenize_b200 import _lib as L

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peak, peak_src = measured_hbm_peak()

    d0, d1 = workload.shard_range(args.pairs, rank, world)          # shard by document, no collective
    n = d1 - d0
    tok = Tokenize(devices=[local_rank])
    tok.set_option("max_chunk_bytes", max(1 << 27, 1 << int(np.ceil(np.log2(args.chunk * 112.0)))))   # both sides of a chunk (~106 MB per 1M pairs)
    for kv in os.environ.get("GENZTOK_OPTIONS", "").split(","):      # e.g. GENZTOK_OPTIONS=rows_minb=6 (experiments)
        if "=" in kv:
            tok.set_option(kv.split("=")[0], int(kv.split("=")[1]))
    t_setup = time.perf_counter()
    S = Stream(tok, torch, dev, d0, n, args.chunk)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup
    n_chunks = len(S.calls)

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.busy = True

    # ---- pass 0 (untimed as a step): cold word cache; digest of every plane; token count; no ValueError rows -----------
    S.encode(0)                                                     # (the library's work areas are allocated by the first call: not part of "cold")
    torch.cuda.synchronize()
    tok.cache_reset()
    acc = torch.zeros(1, dtype=torch.int64, device=dev)
    tok_acc = torch.zeros(1, dtype=torch.int64, device=dev)
    bad_acc = torch.zeros(1, dtype=torch.int64, device=dev)
    cold_ev = []
    for c in range(n_chunks):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = S.encode(c)
        b.record()
        cold_ev.append((a, b))
        tok.digest_device(out, d0 + S.calls[c][5], acc)
        tok_acc += out["row_len"].sum(dtype=torch.int64)
        bad_acc += out["row_status"].sum(dtype=torch.int64)
    torch.cuda.synchronize()
    tok.check_errors(dev)
    cold_ms = [a.elapsed_time(b) for a, b in cold_ev]
    tokens_per_step = int(tok_acc.item())
    digest = int(acc.item()) & 0xFFFFFFFFFFFFFFFF
    assert int(bad_acc.item()) == 0, "rows the reference would reject in a clean batch"

    # ---- warm-up, then K timed passes --------------------------------------------------------------------------------
    for _ in range(args.warmup):
        S.run_pass()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = tok.launch_count()
    step_ms = timed_passes(torch, S.run_pass, args.steps)
    if world > 1:
        dist.barrier()
    launches = tok.launch_count() - launches0
    dev_ms = float(sum(step_ms))
    tok.check_errors(dev)
    if args.dump_outputs and rank == 0:                              # before anything else overwrites the reused planes
        dump_outputs(S.calls[-1][2], d0 + S.calls[-1][5], args.dump_outputs)

    # ---- per-kernel durations (library-side CUDA events on the launching stream), outside the timed region ---------------
    prof_chunks = list(range(min(n_chunks, 8)))
    tok.set_profiling(True)
    tok.profile_report(reset=True)
    S.run_pass(prof_chunks)
    torch.cuda.synchronize()
    prof = tok.profile_report(reset=True)
    tok.set_profiling(False)
    kernels = kernel_table(prof, len(prof_chunks), peak)
    warm_chunk_ms = float(np.mean(timed_passes(torch, lambda: S.encode(0), 5)))

    # ---- arms: cold cache, 1 % adversarial words ----------------------------------------------------------------------
    arms = None
    if not args.no_arms:
        arms = {"cold": {"what": "pass 0: the first pass over the share after genztok_cache_reset (every word of the first chunks goes through k_bpe_pending)",
                         "first_chunk_ms": cold_ms[0], "pass_ms": float(sum(cold_ms)), "warm_chunk_ms": warm_chunk_ms,
                         "first_chunk_cold_over_warm": cold_ms[0] / warm_chunk_ms if warm_chunk_ms else None,
                         "pass_cold_over_warm": float(sum(cold_ms)) / (dev_ms / args.steps) if dev_ms else None}}
        nn = min(n, 8 * args.chunk)
        nc = max(1, ((nn + args.chunk - 1) // args.chunk) // 2)
        NS = Stream(tok, torch, dev, d0, nn, args.chunk, noise=0.01, seed=SEED + 1, planes=S.planes)
        first, second = list(range(0, nc)), list(range(nc, len(NS.calls))) or list(range(0, nc))
        NS.run_pass(first)                                        # vocabulary warm; the noise words of the timed chunks are new
        torch.cuda.synchronize()
        tok.set_profiling(True)
        tok.profile_report(reset=True)
        ms = timed_passes(torch, lambda: NS.run_pass(second), 1)[0]
        nprof = tok.profile_report(reset=True)
        tok.set_profiling(False)
        ntok = 0
        for c in second:
            ntok += int(NS.encode(c)["row_len"].sum().item())
        nalg = NS.alg_bytes(second)
        arms["noise"] = {"what": "1 %% of the words replaced by adversarial ones (glued words, random strings, vocab-only punctuation, '\\n'-attached, exotic "
                                 "whitespace, markers, long tokens): %d chunks with fresh noise words after %d warm-up chunks, word cache warm for the vocabulary" % (len(second), len(first)),
                         "noise": 0.01, "pairs": sum(NS.calls[c][0].numel() - 1 for c in second), "ms": ms, "tokens_per_s": ntok / (ms * 1e-3),
                         "alg_gb_per_s": nalg / (ms * 1e-3) / 1e9, "hbm_frac": nalg / (ms * 1e-3) / 1e9 / peak,
                         "kernels": kernel_table(nprof, len(second), peak)}
        tok.check_errors(dev)
        del NS

    # ---- end-to-end leg: public API, host buffers, copies inside the timed region ----------------------------------------
    import ctypes as C
    lib = L.load()
    ne = min(n, args.e2e_pairs)
    e2e_ms, h2d, d2h, e2e_tokens = 0.0, 0, 0, 0
    if args.e2e_steps > 0 and ne > 0:
        cuts = torch.stack([S.toff[ne], S.poff[ne]]).cpu().tolist()
        offs = [S.toff[:ne + 1].cpu().numpy(), S.poff[:ne + 1].cpu().numpy()]
        pins, hps = [], []
        for src, nb in ((S.text, cuts[0]), (S.pair, cuts[1])):
            hp = lib.genztok_host_alloc(nb + 64)
            hps.append(hp)
            buf = np.frombuffer((C.c_uint8 * nb).from_address(hp), dtype=np.uint8)
            buf[:] = src[:nb].cpu().numpy()
            pins.append(buf)
        for i in range(args.e2e_steps + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            be = tok.encode_batch((pins[0], offs[0]), (pins[1], offs[1]), max_len=MAX_LEN, sequence_id=False)
            checksum = int(be["row_len"][-1])                     # the result is in host memory when the call returns
            dt = time.perf_counter() - t0
            if i > 0:
                e2e_ms += dt * 1e3
            h2d = int(cuts[0] + cuts[1]) + offs[0].nbytes + offs[1].nbytes
            d2h = int(getattr(be, "d2h_bytes", 0)) or (be["input_ids"].nbytes + be["attention_mask"].nbytes + be["token_type_ids"].nbytes + be["row_len"].nbytes * 2 + ne)
            e2e_tokens = int(be["real_tokens"])
            del be
        for hp in hps:
            lib.genztok_host_free(hp)
        del pins

    # ---- what the box gives all ranks at once over PCIe (the ceiling of the end-to-end leg; tools/pcie_probe.py is the long form) ----
    box = None
    if args.e2e_steps > 0 and ne > 0:
        box = pcie_box_probe(torch, dist, world, dev)

    # ---- side measurements (N = 1 only; reported under "extra", not the headline) ------------------------------------------
    extra = None
    if world == 1 and not args.no_extras:
        extra = run_extras(torch, tok, S, dev, peak, workload, Tokenize)

    clocks = sampler.stop()
    # ---- max over ranks ------------------------------------------------------------------------------------------------------
    t = torch.tensor([dev_ms, e2e_ms] + step_ms, dtype=torch.float64, device=dev)
    s = torch.tensor([tokens_per_step, S.in_bytes, launches, e2e_tokens, S.alg_bytes(), n, ne], dtype=torch.float64, device=dev)
    dg = torch.tensor([digest - (1 << 64) if digest >= (1 << 63) else digest], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        parts = [torch.zeros_like(dg) for _ in range(world)]
        dist.all_gather(parts, dg)
        digest = sum(int(p.item()) for p in parts) & 0xFFFFFFFFFFFFFFFF
    tl = t.tolist()
    dev_ms, e2e_ms, step_ms = float(tl[0]), float(tl[1]), [float(x) for x in tl[2:]]
    tot_tokens, tot_in_bytes, tot_launches, tot_e2e_tokens, tot_alg, tot_pairs, tot_e2e_pairs = [float(x) for x in s.tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = dev_ms / args.steps
    value = tot_tokens / (ms_per_step * 1e-3)
    alg_gbs = tot_alg / (ms_per_step * 1e-3) / 1e9
    dom = max(kernels, key=lambda k: kernels[k]["ms"] * kernels[k]["launches"]) if kernels else None
    dk = kernels.get(dom, {}) if dom else {}
    kernels_ms_per_chunk = sum(v["ms"] * v["launches"] for v in kernels.values())
    traffic, traffic_note = None, "no capture on file for this build"
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("source_hash") == source_hash():
            traffic = tj.get("kernels", {}).get(dom, {}).get("dram_bytes_per_launch")
            traffic_note = tj.get("note", "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch")
        else:
            traffic_note = "profiles/roofline_traffic.json was captured on another build of the kernels: not reported"
    except Exception:
        pass
    e2e_step_ms = e2e_ms / max(args.e2e_steps, 1)
    line = {
        "metric": "encode_tokens_per_sec", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
        "config": {"workload": workload_name(args.pairs), "max_len": MAX_LEN, "pairs_global": args.pairs, "pairs_per_gpu": n, "chunk_pairs": args.chunk,
                   "chunks_per_gpu_per_step": n_chunks, "sharding": "by document, contiguous ranges, no collective on the data path",
                   "l2": "not flushed: every chunk reads ~106 MB of text and writes 1.6 GB of planes, the 126 MB L2 holds neither; the word cache and tables are meant to stay in L2",
                   "outputs": "input_ids int32 + attention_mask uint8 + token_type_ids int8 [chunk,256] + row_len / seq_len / row_status, one reused set of planes",
                   "generator": "workload.generate_hashed on the device (csrc/synth.cuh), seed %d; untimed set-up %.1f s" % (SEED, setup_s)},
        "pairs_per_s": tot_pairs / (ms_per_step * 1e-3),
        "input_gb_per_s": tot_in_bytes / (ms_per_step * 1e-3) / 1e9,
        "alg_gb_per_s": alg_gbs,
        "hbm_frac_of_step": alg_gbs / (world * peak),
        "step_ms": {"mean": ms_per_step, "median": float(np.median(step_ms)), "best": float(min(step_ms)), "worst": float(max(step_ms)), "timed_region_s": dev_ms * 1e-3},
        "digest": {"planes_u64": "%016x" % digest, "what": "order-independent digest of input_ids / attention_mask / token_type_ids of all %d pairs (k_plane_digest, pass 0): "
                                                           "the same at every GPU count" % args.pairs, "real_tokens": int(tot_tokens)},
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": dk.get("alg_gb_per_s"), "peak": peak, "unit": "GB/s",
                     "frac": dk.get("frac_of_peak"), "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                     "alg_bytes_per_launch": dk.get("alg_bytes"), "kernel_ms": dk.get("ms"), "kernel_launches_per_chunk": dk.get("launches"),
                     "kernels_ms_per_chunk": kernels_ms_per_chunk,
                     "kernel_share_of_step": dk.get("ms", 0) * dk.get("launches", 0) / kernels_ms_per_chunk if kernels_ms_per_chunk else None,
                     "frac_of_nominal_8TBs": (dk.get("alg_gb_per_s") or 0) / NOMINAL_HBM_GBS,
                     "whole_path": {"alg_bytes_per_step": tot_alg, "bytes_per_pair": tot_alg / tot_pairs if tot_pairs else None, "achieved": alg_gbs,
                                    "frac": alg_gbs / (world * peak), "frac_of_nominal_8TBs": alg_gbs / (world * NOMINAL_HBM_GBS),
                                    "frac_best_step": tot_alg / (min(step_ms) * 1e-3) / 1e9 / (world * peak),
                                    "note": "all kernels and launch gaps of a step against n_gpus x peak: the number to compare with the 50% target"}},
        "e2e": {"value": tot_e2e_tokens / (e2e_step_ms * 1e-3) if e2e_ms else None, "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_step_ms, "pairs_per_step_per_gpu": ne, "d2h_gb_per_s_per_rank": d2h / (e2e_step_ms * 1e-3) / 1e9 if e2e_ms else None,
                "api": "Tokenize.encode_batch(packed pairs in pinned host memory) -> pinned numpy planes; a bounded share (%d pairs per GPU) of the batch per step" % ne,
                "box_pcie": box},
        "gpu_launches": int(tot_launches),
        "clocks": clocks,
        "kernels": kernels,
    }
    if arms is not None:
        line["arms"] = arms
    if extra is not None:
        line["extra"] = extra
    if not args.no_cpu and world == 1:            # the CPU baseline is reported at N=1 only
        try:
            line["cpu_baseline"] = cpu_baseline_block()
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": host_threads(), "kind": "reference", "sample": "failed: %r" % (e,)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def pcie_box_probe(torch, dist, world, dev, mb=256, reps=4):
    """Plain pinned-memory copies by every rank at once: device->host alone, and both directions together (GB/s per direction)."""
    h_out = torch.empty(mb << 20, dtype=torch.uint8).pin_memory()
    h_in = torch.zeros(mb << 20, dtype=torch.uint8).pin_memory()
    d_a = torch.zeros(mb << 20, dtype=torch.uint8, device=dev)
    d_b = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def leg(both):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            with torch.cuda.stream(s1):
                h_out.copy_(d_a, non_blocking=True)
            if both:
                with torch.cuda.stream(s2):
                    d_b.copy_(h_in, non_blocking=True)
        torch.cuda.synchronize()
        return reps * (mb << 20) / (time.perf_counter() - t0) / 1e9

    leg(True)
    v = torch.tensor([leg(False), leg(True)], dtype=torch.float64, device=dev)
    lo = v.clone()
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    return {"d2h_gb_per_s_all_ranks": float(v[0]), "d2h_gb_per_s_slowest_rank": float(lo[0]),
            "both_directions_gb_per_s_per_direction_all_ranks": float(v[1]), "both_directions_slowest_rank": float(lo[1]),
            "what": "cudaMemcpyAsync of %d MiB pinned buffers by all %d ranks at once: the ceiling the host side of this box puts on the end-to-end leg" % (mb, world)}


def run_extras(torch, tok, S, dev, peak, workload, Tokenize):
    """BASELINE configs[1], [3], [4] at one GPU (side measurements)."""
    extra = {}
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def timed(fn, reps=5, warm=2):
        for _ in range(warm):
            flush.zero_(); fn()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs:
            flush.zero_(); a.record(); fn(); b.record()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    # configs[3]: decode of the encoded planes, streamed through a reused text ring
    ncd = min(len(S.calls), 8)
    ring, dms, dms_read, dbytes, rows = None, 0.0, 0.0, 0, 0
    for rep in range(3):                                            # 0: sizes the ring; 1: timed with the size read back per chunk; 2: timed without any host read
        for c in range(ncd):
            out = S.encode(c)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            txt, toff = tok.decode_device(out["input_ids"], out=ring, sync=rep < 2)
            b.record()
            if rep == 0 and (ring is None or ring.numel() < txt.numel()):
                ring = torch.empty((int(txt.numel() * 1.03) + (1 << 20),), dtype=torch.uint8, device=dev)
            torch.cuda.synchronize()
            if rep == 1:
                dms_read += a.elapsed_time(b); dbytes += int(txt.numel()); rows += out["input_ids"].shape[0]
            if rep == 2:
                dms += a.elapsed_time(b)
    dalg = 4 * rows * MAX_LEN + dbytes + 16 * rows
    extra["configs3_decode_256"] = {"workload": "decode of the [chunk,256] input_ids planes of configs[2] (pads print as '<pad>'), %d chunks streamed into a reused text ring" % ncd,
                                    "rows": rows, "ms": dms, "rows_per_s": rows / (dms * 1e-3), "ids_per_s": rows * MAX_LEN / (dms * 1e-3), "text_bytes": dbytes,
                                    "alg_gb_per_s": dalg / (dms * 1e-3) / 1e9, "hbm_frac": dalg / (dms * 1e-3) / 1e9 / peak,
                                    "ms_with_size_read": dms_read, "hbm_frac_with_size_read": dalg / (dms_read * 1e-3) / 1e9 / peak,
                                    "note": "both passes (lengths + write) per chunk through genztok_decode_device_into: no host read between them (the kernels check that "
                                            "the text fits the ring); ms_with_size_read: the same with the text size read back after every chunk"}
    del ring
    # configs[1]: 1,048,576 single sentences, max_len 128
    n1, W1 = 1 << 20, 128
    t1, o1, b1 = tok.synth_device(SEED, 0, n1, 0, LO, HI, 0.0, device=dev)
    out1 = {"input_ids": torch.empty((n1, W1), dtype=torch.int32, device=dev), "attention_mask": torch.empty((n1, W1), dtype=torch.uint8, device=dev),
            "row_len": torch.empty((n1,), dtype=torch.int32, device=dev)}
    f1 = lambda: tok.encode_device(t1, o1, max_len=W1, out=out1, text_bytes=b1)
    ms = timed(f1)
    tok.cache_reset()
    cold = timed(f1, reps=1, warm=0)[0]
    alg1 = b1 + 8 * (n1 + 1) + n1 * W1 * 5
    toks1 = int(out1["row_len"].sum().item())
    extra["configs1_singles_128"] = {"workload": "1,048,576 single sentences, max_len=128, ids + mask (BASELINE configs[1]); L2 flushed between steps",
                                     "ms": float(np.mean(ms)), "ms_best": float(min(ms)), "tokens_per_s": toks1 / (float(np.mean(ms)) * 1e-3),
                                     "alg_gb_per_s": alg1 / (float(np.mean(ms)) * 1e-3) / 1e9, "hbm_frac": alg1 / (float(np.mean(ms)) * 1e-3) / 1e9 / peak,
                                     "cold_ms": cold, "cold_over_warm": cold / float(np.mean(ms))}
    holder = {}
    dms1a = float(np.mean(timed(lambda: holder.__setitem__("d", tok.decode_device(out1["input_ids"])))))
    db1 = int(holder["d"][0].numel())
    ring1 = torch.empty((db1 + (1 << 20),), dtype=torch.uint8, device=dev)
    dms1 = float(np.mean(timed(lambda: tok.decode_device(out1["input_ids"], out=ring1, sync=False))))
    dalg1 = 4 * n1 * W1 + db1 + 16 * n1
    extra["configs1_decode_128"] = {"workload": "decode of the [1M,128] planes of configs[1] into a reused text buffer; L2 flushed between steps", "ms": dms1,
                                    "rows_per_s": n1 / (dms1 * 1e-3), "text_bytes": db1,
                                    "alg_gb_per_s": dalg1 / (dms1 * 1e-3) / 1e9, "hbm_frac": dalg1 / (dms1 * 1e-3) / 1e9 / peak,
                                    "ms_alloc_and_size_read": dms1a, "hbm_frac_alloc_and_size_read": dalg1 / (dms1a * 1e-3) / 1e9 / peak,
                                    "note": "ms: genztok_decode_device_into, no host read; ms_alloc_and_size_read: the two-step protocol with the text tensor allocated per call"}
    del ring1
    # the reference's DEFAULT call shape (tokenize.py:184-190: max_len=None -> no padding, no truncation): ragged rows through the
    # host API (there is no padded plane to hold them on the device); kernels by the library's CUDA events, the call by wall clock
    import ctypes as C
    from genz_tokenize_b200 import _lib as L
    hp1 = L.load().genztok_host_alloc(b1 + 64)                      # the caller's text in pinned memory, as in the e2e leg
    ht1 = np.frombuffer((C.c_uint8 * b1).from_address(hp1), dtype=np.uint8)
    ht1[:] = t1[:b1].cpu().numpy()
    h1 = (ht1, o1.cpu().numpy())
    tok.encode_batch(h1)                                            # allocations
    calls = []
    for _ in range(4):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        rg = tok.encode_batch(h1)
        calls.append((time.perf_counter() - t0) * 1e3)
        rtok = int(rg["real_tokens"]); rd2h = int(rg.d2h_bytes); del rg
    call_ms = float(np.median(calls))
    tok.set_profiling(True); tok.profile_report(reset=True)
    rg = tok.encode_batch(h1)
    rprof = tok.profile_report(reset=True); tok.set_profiling(False)
    ralg = b1 + 8 * (n1 + 1) + 5 * rtok + 8 * (n1 + 1)              # SURVEY.md 8 d4, ragged: utf8 + offsets in, 5 B per token + row offsets out
    rk_ms = sum(v["ms"] for v in rprof.values())
    extra["default_call_ragged"] = {"workload": "the 1,048,576 single sentences with max_len=None (ragged rows: ids + mask + int64 row offsets), Tokenize.encode_batch, "
                                                "pinned host text in, pinned host rows out",
                                    "kernels_ms": rk_ms, "call_ms": call_ms, "call_ms_all": [round(c, 2) for c in calls], "tokens_per_s_kernels": rtok / (rk_ms * 1e-3),
                                    "tokens_per_s_call": rtok / (call_ms * 1e-3), "alg_gb_per_s_kernels": ralg / (rk_ms * 1e-3) / 1e9,
                                    "hbm_frac_kernels": ralg / (rk_ms * 1e-3) / 1e9 / peak, "h2d_bytes": int(b1 + 8 * (n1 + 1)), "d2h_bytes": rd2h,
                                    "kernels": {k: round(v["ms"], 4) for k, v in rprof.items() if v["ms"] > 0.005}}
    # configs[1] end to end through the host API: the same sentences, max_len=128, pinned text in, pinned planes out
    tok.encode_batch(h1, max_len=W1)                                # allocations
    calls1 = []
    for _ in range(5):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        be1 = tok.encode_batch(h1, max_len=W1)
        calls1.append((time.perf_counter() - t0) * 1e3)
        e_tok, e_d2h = int(be1["real_tokens"]), int(be1.d2h_bytes); del be1
    c1 = float(np.median(calls1))
    extra["configs1_e2e_host"] = {"workload": "the 1,048,576 single sentences, max_len=128, Tokenize.encode_batch: pinned host text in, pinned [n,128] planes out "
                                              "(only the columns that can differ from padding cross PCIe)",
                                  "call_ms": c1, "call_ms_all": [round(c, 2) for c in calls1], "tokens_per_s": e_tok / (c1 * 1e-3),
                                  "h2d_bytes": int(b1 + 8 * (n1 + 1)), "d2h_bytes": e_d2h, "d2h_gb_per_s": e_d2h / (c1 * 1e-3) / 1e9}
    del ht1, h1
    L.load().genztok_host_free(hp1)
    del rg, t1, o1, holder
    # configs[4]: custom vocab / merges, long documents, max_len 4096, low word reuse -- reported cold (its definition) and warm
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        vp, mp, words = workload.build_custom_model(td)
        tok5 = Tokenize.fromFile(vp, mp, devices=[dev.index])
        tok5.set_option("max_chunk_bytes", 1 << 28)
        nd5, W5 = 1024, 4096
        b5, o5 = workload.long_documents(words, nd5)
        d5 = torch.from_numpy(np.concatenate([b5, np.zeros(64, dtype=np.uint8)])).to(dev)
        do5 = torch.from_numpy(o5).to(dev)
        out5 = {"input_ids": torch.empty((nd5, W5), dtype=torch.int32, device=dev), "attention_mask": torch.empty((nd5, W5), dtype=torch.uint8, device=dev),
                "row_len": torch.empty((nd5,), dtype=torch.int32, device=dev)}
        f5 = lambda: tok5.encode_device(d5, do5, max_len=W5, out=out5, text_bytes=int(o5[-1]))
        f5(); torch.cuda.synchronize()                             # allocations
        colds = []
        for _ in range(3):
            tok5.cache_reset()
            colds.append(timed(f5, reps=1, warm=0)[0])
        warm = timed(f5, reps=5, warm=1)
        alg5 = int(o5[-1]) + 8 * (nd5 + 1) + nd5 * W5 * 5
        extra["configs4_custom_vocab_long_docs"] = {
            "workload": "Tokenize.fromFile, %d-word custom vocab with a merge chain per word, %d documents of 6-9 k uniformly sampled words (%.0f KB each), max_len=4096 "
                        "(BASELINE configs[4]: heavy truncation, low word reuse)" % (len(words), nd5, o5[-1] / nd5 / 1e3),
            "cold_ms": float(np.mean(colds)), "warm_ms": float(np.mean(warm)), "cold_docs_per_s": nd5 / (float(np.mean(colds)) * 1e-3),
            "warm_docs_per_s": nd5 / (float(np.mean(warm)) * 1e-3), "cold_over_warm_throughput": float(np.mean(warm)) / float(np.mean(colds)),
            "cold_alg_gb_per_s": alg5 / (float(np.mean(colds)) * 1e-3) / 1e9, "warm_alg_gb_per_s": alg5 / (float(np.mean(warm)) * 1e-3) / 1e9,
            "real_tokens": int(out5["row_len"].sum().item())}
        del tok5
    return extra


if __name__ == "__main__":
    sys.dont_write_bytecode = True       # the tree this runs from may be read-only, and a run leaves nothing in it
    main()
