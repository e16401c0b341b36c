#!/usr/bin/env python3
"""bench.py -- the reference's headline metric on B200 (BASELINE.json): BPE train merges/s (+ wall-s) on a 1 GiB
synthetic Zipfian UTF-8 corpus at vocab 32768 (configs[2]) and encode MB/s of 10 GiB of synthetic text with that
model (configs[3]), at 1/2/4/8 GPUs; configs[4] (8 GiB, vocab 100000) with --config5 (default at 8 GPUs).

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (GPU)
    python bench.py --impl reference [...]                         the reference's own CPU code, bounded sample

Every timed leg runs exactly K timed steps. --dump-outputs DIR: after the timed steps, rank 0 writes what each timed leg
computed in its last step as DIR/<name>.npy in float64 (exact for ids, counts and bytes): train_merges, train_counts,
train_<other mode>_merges / _counts, encode_ids (the ids of the last encode batch), decode_bytes, config5_merges. An
array of more than DUMP_ROWS rows is cut to a fixed, seeded sample of its rows, kept in order. The inputs depend on the
arguments alone (seeded generators), so two builds can be compared file by file.

One JSON line on stdout (rank 0). PyTorch is plumbing only: torch.distributed (NCCL) barrier / max over ranks, device
buffers, streams and events. All compute goes through the C ABI of libminbpe_b200.so (include/minbpe_b200.h).

What a "step" is, and what N > 1 means (strong scaling: the workload is the same at every N):
  train   one complete merge loop (vocab-256 merges) over the deduplicated corpus resident in HBM.
          N = 1: mbpe_trainer_run. N > 1: the SHARDED trainer (mbpe_sharded_trainer_run) -- the unique chunks of the
          same corpus are sharded over the ranks, every rank keeps a replica of the pair table, per-merge exchange of
          the count deltas over NVLink. (N independent replicas are reported beside it as train.replicas, not as value.)
  encode  BASELINE config 4: --encode-gib (10) DISTINCT GiB of text, cut into contiguous ranges of whole chunks over the
          ranks (mbpe_plan_shards), every rank streams its range ONCE through an encoder whose caches start empty.
  decode  ids of one batch -> bytes (resident).
Every leg is diffed: train against the CPU oracle at full size (and against the compiled reference on a sample), encode
against the compiled reference's id stream on a >= 256 MiB slice and by decode(encode(x)) == x.
"""
import argparse
import hashlib
import importlib.util
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED_TRAIN, SEED_ENCODE, SEED_CONFIG5, SEED_DUMP = 0x5EED0001, 0x5EED0002, 0x5EED0003, 0x5EED00D0
MIB = 1 << 20
DUMP_ROWS = 1 << 19  # per array: the seven arrays of --dump-outputs stay under 64 MiB in float64


def dump_rows(n):
    """indices of the rows --dump-outputs keeps of an n-row array: all of them, or a fixed seeded sample in order"""
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(SEED_DUMP).choice(n, DUMP_ROWS, replace=False))


def write_outputs(d, arrays):
    os.makedirs(d, exist_ok=True)
    for name, x in arrays.items():
        x = np.asarray(x)
        np.save(os.path.join(d, name + ".npy"), x[dump_rows(len(x))].astype(np.float64))


def load_pkg():
    spec = importlib.util.spec_from_file_location("minbpe_cc_b200", os.path.join(ROOT, "minbpe-cc_b200", "__init__.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["minbpe_cc_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json), or None"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(kernel)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed regions."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        self.marks = []

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self, t0, t1):
        self.marks.append((t0, t1))

    def summary(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if self.marks and not any(a - 0.2 <= t <= b + 0.2 for a, b in self.marks):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def safe_prefix(text: bytes, n: int) -> bytes:
    """largest prefix <= n bytes ending at a regex-safe cut: after '\\n', before a printable ASCII byte (SURVEY H7)."""
    n = min(n, len(text))
    lo = max(0, n - 65536)
    last = None
    for m in re.finditer(rb"\n[\x21-\x7e]", text[lo:n]):
        last = m
    return text[:lo + last.start() + 1] if last else text[:n]


# --------------------------------------------------------------------------------------------------------
# the reference's own CPU implementation (oracle/_ref/ref_driver = reference headers compiled verbatim) on bounded
# samples of the same workloads. Input text comes from oracle/_ref/synthgen (the generator as a stand-alone program):
# nothing of the product library is loaded by the reference arm.
# --------------------------------------------------------------------------------------------------------
def synth_text(seed, n_bytes):
    from oracle import oracle as O
    gen = os.path.join(os.path.dirname(O.REF_DRIVER), "synthgen")
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "t.bin")
        subprocess.check_call([gen, hex(seed), str(n_bytes), p])
        return open(p, "rb").read()


def ref_train_sample(sample_mib, n_merges, mode, workload_bytes):
    from oracle import oracle as O
    text = safe_prefix(synth_text(SEED_TRAIN, sample_mib * MIB), sample_mib * MIB)  # blockwise generator: same first MiBs
    with tempfile.TemporaryDirectory() as td:
        inp, model = os.path.join(td, "in.txt"), os.path.join(td, "m.model")
        open(inp, "wb").write(text)
        if os.path.exists(O.REF_DRIVER):
            kind = "reference"
            p = subprocess.run([O.REF_DRIVER, "train", inp, model, str(256 + n_merges), "gpt4", mode],
                               capture_output=True, text=True)
            secs = float(re.search(r"REF_TIME_S ([0-9.eE+-]+)", p.stderr).group(1))
            merges = O.read_model(model)[2]
        else:  # the compiled reference did not travel: time the C restatement's literal walk instead
            kind = "port"
            t0 = time.time()
            t, o, w = O.flatten(O.chunks_of(text, "gpt4"), dedup=False)
            merges, _ = O.train(t, o, w, 256 + n_merges, mode, impl="rescan")
            secs = time.time() - t0
    mps = n_merges / secs
    return {"value": mps, "unit": "merges/s", "cores": 1, "kind": kind,
            "sample": f"Tokenizer::train (regex split + lists + merge loop) on the first {len(text)} bytes "
                      f"({sample_mib} MiB) of the same synthetic corpus, {n_merges} merges, {mode}, 1 thread "
                      f"(the reference is single-threaded); took {secs:.2f} s",
            "seconds": secs, "sample_bytes": len(text), "sample_merges": n_merges,
            "value_extrapolated_to_workload": mps * len(text) / float(workload_bytes),
            "extrapolation": "per-merge cost of the reference is linear in corpus bytes (it walks every chunk every "
                             "merge, Tokenizer.h:309-320): merges/s x sample_bytes / workload_bytes",
            }, merges, text


def ref_encode_sample(model_path, sample_mib):
    from oracle import oracle as O
    text = safe_prefix(synth_text(SEED_ENCODE, sample_mib * MIB), sample_mib * MIB)
    with tempfile.TemporaryDirectory() as td:
        inp, out = os.path.join(td, "in.txt"), os.path.join(td, "o.enc")
        open(inp, "wb").write(text)
        if os.path.exists(O.REF_DRIVER):
            kind = "reference"
            p = subprocess.run([O.REF_DRIVER, "encode", inp, model_path, out], capture_output=True, text=True)
            secs = float(re.search(r"REF_TIME_S ([0-9.eE+-]+)", p.stderr).group(1))
            enc = open(out, "rb").read()
        else:
            kind = "port"
            pat, sp, m = O.read_model(model_path)
            t0 = time.time()
            enc = O.encode_text(text, pat, sp, m).tobytes()
            secs = time.time() - t0
    return {"value": len(text) / 1e6 / secs, "unit": "MB/s", "cores": 1, "kind": kind,
            "sample": f"Tokenizer::encode (regex split + merge scan) on the first {len(text)} bytes ({sample_mib} MiB) of "
                      f"the synthetic encode corpus, cut at a regex-safe point, 1 thread; took {secs:.2f} s",
            "seconds": secs, "sample_bytes": len(text), "n_ids": len(enc) // 4,
            "sha256": hashlib.sha256(enc).hexdigest()}, text


def reference_full_run_record():
    """SURVEY 8(d): the un-extrapolated ratio -- a FULL 32k-vocab reference run on a 16 MiB slice takes the reference
    about an hour, so it is run once per round (tools/ref_full_16mib.py) and its record is committed."""
    p = os.path.join(ROOT, "profiles", "reference_full_16MiB.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


def run_reference_arm(a, rank):
    if rank != 0:
        return
    vals = []
    for _ in range(a.warmup + a.steps):
        cb, merges, _ = ref_train_sample(a.ref_sample_mib, a.ref_merges, a.mode, a.corpus_mib * MIB)
        vals.append(cb)
    if a.dump_outputs:
        write_outputs(a.dump_outputs, {"train_merges": merges})
    vals = vals[a.warmup:] or vals
    v = sum(x["value"] for x in vals) / len(vals)
    cb = dict(vals[-1], value=v)
    cfg = workload_config(a)
    # what this arm really ran (the full workload would take the reference > 100 CPU-hours and ~47 GB, SURVEY 6.2)
    cfg.update({"sample_of_workload": True, "sample_bytes": cb["sample_bytes"], "sample_merges": cb["sample_merges"],
                "same_config_as_gpu_arm": False,
                "comparable_value": "cpu_baseline.value_extrapolated_to_workload (merges/s at the full corpus size)"})
    line = {"impl": "reference", "metric": "bpe_train_merges_per_sec", "value": v, "unit": "merges/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * cb["seconds"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": cfg, "cpu_baseline": cb,
            "e2e": {"value": v, "unit": "merges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "reference_full_16MiB_run": reference_full_run_record()}
    print(json.dumps(line))


def workload_config(a):
    return {"workload": f"train {a.corpus_mib} MiB synthetic Zipfian UTF-8 corpus (seed 0x{SEED_TRAIN:X}), "
                        f"--vocab-size {a.vocab} --encoder gpt4 -c {a.mode}",
            "vocab_size": a.vocab, "corpus_bytes": a.corpus_mib * MIB, "mode": a.mode, "encoder": "gpt4",
            "engine": a.engine, "l2": "each step re-streams the whole working set (> L2) and a 256 MiB buffer is "
                                      "written between timed steps"}


# --------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--corpus-mib", type=int, default=1024)
    ap.add_argument("--vocab", type=int, default=32768)
    ap.add_argument("--mode", default="lexical", choices=["first", "lexical"])
    ap.add_argument("--engine", default="persistent", choices=["persistent", "stepwise"])
    ap.add_argument("--encode-gib", type=float, default=10.0, help="config 4: distinct text streamed once, all ranks together")
    ap.add_argument("--encode-batch-mib", type=int, default=1024, help="resident batch size (a device batch is < 4 GiB)")
    ap.add_argument("--ref-sample-mib", type=int, default=4)
    ap.add_argument("--ref-merges", type=int, default=128)
    ap.add_argument("--ref-encode-mib", type=int, default=256)
    ap.add_argument("--skip-encode", action="store_true")
    ap.add_argument("--skip-first", action="store_true", help="skip the first-occurrence-mode train line")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--config5", action="store_true", help="also run config 5 (8 GiB, vocab 100000); default at 8 GPUs")
    ap.add_argument("--config5-gib", type=int, default=8)
    ap.add_argument("--config5-vocab", type=int, default=100000)
    ap.add_argument("--selftest", action="store_true", help="N > 1: diff the sharded trainer against the oracle on the goldens first")
    ap.add_argument("--no-check", action="store_true", help="skip the full-size diff of the merge list against the CPU oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of every leg as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference_arm(a, rank)
        return

    import torch
    import torch.distributed as dist

    pkg = load_pkg()
    if pkg.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libminbpe_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream().cuda_stream
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gpt4 = pkg.patterns()["gpt4"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def all_true(flag):
        if world == 1:
            return bool(flag)
        t = torch.tensor([int(bool(flag))], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def bcast(ident):
        t = torch.from_numpy(ident.copy()).to(dev)
        dist.broadcast(t, 0)
        return t.cpu().numpy()

    clocks = ClockSampler(local_rank) if rank == 0 else None
    peak, peak_src = measured_peaks()
    comm = pkg.Comm(rank, world, local_rank, bcast) if world > 1 else None

    def timed_steps(fn, n_warm, n_steps):
        """fn() enqueues one step on the current stream; device time per step (CUDA events), L2 flushed between steps,
        barrier + synchronize on both sides of the timed region, max over ranks"""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * (n_warm + n_steps))]
        out, wall0 = None, time.time()
        for i in range(n_warm + n_steps):
            flush_buf.fill_(i & 0xFF)
            if i == n_warm:
                barrier()
                wall0 = time.time()
            ev[2 * i].record()
            out = fn()
            ev[2 * i + 1].record()
        barrier()
        if clocks:
            clocks.mark(wall0, time.time())
        ms = [ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(n_warm, n_warm + n_steps)]
        return max_over_ranks(sum(ms) / len(ms)), out

    # ---------------- optional: sharded-trainer parity on the golden fixtures, where the scaling run can see it ------
    selftest = None
    if world > 1 and a.selftest:
        from oracle import oracle as O
        selftest = {}
        for name in ("taylorswift.txt", "sample.txt"):
            text_g = open(os.path.join(ROOT, "tests", "golden", "data", name), "rb").read()
            s, e = pkg.split(gpt4, text_g)
            tg, og, wg = pkg.dedup(text_g, s, e)
            for mode in ("first", "lexical"):
                om, oc = O.train(tg, og, wg, 512, mode)
                sm, sc, _ = comm.train(tg, og, wg, 512, mode, stream)
                selftest[f"{name}/{mode}"] = all_true(sm.shape == om.shape and bool((sm == om).all()) and bool((sc == oc).all()))

    # ---------------- host prep (outside every timed region): corpus, regex split, dedup -----------------
    t0 = time.time()
    text = pkg.synth_corpus(SEED_TRAIN, a.corpus_mib * MIB)  # every rank holds the same corpus; N > 1 shards its unique chunks
    t_gen = time.time() - t0
    tb = text.tobytes()
    t0 = time.time()
    tok, off, w, n_chunks = pkg.split_dedup(gpt4, tb)
    t_split = time.time() - t0

    # ---------------- train: device-resident steps -------------------------------------------------------
    if world == 1:
        trainer = pkg.Trainer(tok, off, w, device=local_rank)
        ms_per_step, (merges, counts, stats) = timed_steps(lambda: trainer.run(a.vocab, a.mode, a.engine, stream), a.warmup, a.steps)
        what = "mbpe_trainer_run: one GPU, deduplicated corpus resident"
    else:
        strainer = pkg.ShardedTrainer(comm, tok, off, w)
        ms_per_step, (merges, counts, stats) = timed_steps(lambda: strainer.run(a.vocab, a.mode, stream), a.warmup, a.steps)
        what = (f"mbpe_sharded_trainer_run over {world} GPUs: unique chunks sharded (resident), replicated pair table, "
                "per-merge exchange of count deltas over NVLink")
    dumps = {"train_merges": merges, "train_counts": counts}
    n_done = len(merges)
    value = n_done / (ms_per_step / 1e3)
    model_sha = hashlib.sha256(merges.tobytes()).hexdigest()
    same_everywhere = all_true(True)
    if world > 1:  # every rank must hold the same merge list
        h = torch.tensor(list(hashlib.sha256(merges.tobytes() + counts.tobytes()).digest()), dtype=torch.int32, device=dev)
        h0 = h.clone()
        dist.broadcast(h0, 0)
        same_everywhere = all_true(bool((h == h0).all()))
    launches_train = int(stats["n_launches"]) * a.steps

    line = {
        "metric": "bpe_train_merges_per_sec", "value": value, "unit": "merges/s", "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": workload_config(a),
        "gpu_launches": launches_train,
        "train": {"what": what, "merges": int(n_done), "merges_sha256": model_sha, "gpu_s_per_run": ms_per_step / 1e3,
                  "same_merges_on_every_rank": same_everywhere,
                  "host_prep_s": {"generate": t_gen, "split_dedup": t_split},
                  "n_chunks": int(n_chunks), "n_unique_chunks": int(len(w)), "stats": stats},
    }
    if selftest is not None:
        line["train"]["sharded_selftest_vs_oracle"] = selftest
    # The merge loop is LATENCY-bound: one resident CTA walks a chain of dependent L2 / HBM round trips per merge and
    # moves about a thousand times fewer bytes than a rescan would. `achieved` is still SURVEY 8(d)'s figure (the
    # full-rescan algorithmic volume / device time) so that the number is comparable with the survey's definition;
    # `traffic` is the real DRAM volume of one k_persistent launch from ncu.
    ach = stats["rescan_bytes"] / 1e9 / (ms_per_step / 1e3)
    tr = ncu_traffic("k_persistent")
    line["roofline"] = {"bound": "latency", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                        "traffic": tr["dram_bytes_per_launch"] if tr else None, "traffic_detail": tr,
                        "peak_source": peak_src, "kernel": "k_persistent (+ per-phase grid kernels)",
                        "algorithmic_bytes_per_step": int(stats["rescan_bytes"]),
                        "note": "bound = latency, not HBM: algorithmic bytes = sum over merges of 12*T_m + 16*P_m, what a full "
                                "rescan per merge would move (SURVEY 8(d)); the incremental kernels move ~1000x fewer real "
                                "bytes (traffic), so frac is not a bandwidth utilisation"}

    # ---------------- e2e: reference-facing call, HOST buffers in -> merges out ---------------------------------------
    tk = pkg.Tokenizer(gpt4, device=local_rank)
    tk.set_engine(a.engine)
    if world == 1:
        text_pinned = torch.empty(len(text), dtype=torch.uint8, pin_memory=True)  # the step's input, in pinned host memory
        text_pinned.numpy()[:] = text
        e2e_times = []
        for i in range(1 + a.steps):  # the first call is a warm-up: it sizes the tokenizer's resident device buffers
            barrier()
            t0 = time.time()
            tk.train(text_pinned.numpy(), a.vocab, a.mode)
            torch.cuda.synchronize()
            if i:
                e2e_times.append(time.time() - t0)
        e2e_s = sum(e2e_times) / len(e2e_times)
        st2 = tk.last_train_stats()
        assert hashlib.sha256(tk.merges().tobytes()).hexdigest() == model_sha, "tokenizer path and trainer path disagree"
        on_gpu = bool(st2.get("split_on_gpu"))
        h2d = int(len(tb)) if on_gpu else int(st2["n_positions"] * 4 + (st2["n_unique"] + 1) * 8 + st2["n_unique"] * 4)
        line["e2e"] = {"value": n_done / e2e_s, "unit": "merges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(n_done * 12),
                       "steps": len(e2e_times), "wall_s_per_step": e2e_s, "wall_s_steps": [round(t, 4) for t in e2e_times],
                       "what": "mbpe_tokenizer_train(text) = Tokenizer::train, text in pinned host memory: " +
                               ("H2D text + device split (GPT-4 matcher) + device dedup + merge loop + D2H merges" if on_gpu else
                                "host regex split + dedup + H2D + merge loop + D2H merges"),
                       "split": "device" if on_gpu else "host", "split_dedup_s": st2["split_s"], "gpu_ms": st2["gpu_ms"]}
        # the C-ABI hot-path boundary with deduplicated HOST buffers (H2D + merge loop + D2H per step)
        abi_times = []
        for i in range(a.steps):
            t0 = time.time()
            m2, _, _ = pkg.train(tok, off, w, a.vocab, a.mode, a.engine, device=local_rank)
            abi_times.append(time.time() - t0)
        abi_s = sum(abi_times) / len(abi_times)
        line["e2e_abi"] = {"value": n_done / abi_s, "unit": "merges/s", "wall_s_per_step": abi_s,
                           "what": "mbpe_train(deduplicated host buffers): H2D + merge loop + D2H"}
    else:
        # N > 1: the C-ABI call with HOST buffers -- every rank uploads its shard of the unique chunks inside the call
        e2e_times = []
        for i in range(1 + a.steps):
            barrier()
            t0 = time.time()
            sm, sc, sst = comm.train(tok, off, w, a.vocab, a.mode, stream)
            torch.cuda.synchronize()
            barrier()
            if i:
                e2e_times.append(time.time() - t0)
        e2e_s = max_over_ranks(sum(e2e_times) / len(e2e_times))
        assert hashlib.sha256(sm.tobytes()).hexdigest() == model_sha, "one-shot and resident sharded trainers disagree"
        shard_bytes = int(len(tok) * 4 / world + len(w) * 12 / world)
        line["e2e"] = {"value": n_done / e2e_s, "unit": "merges/s", "h2d_bytes_per_step": shard_bytes, "d2h_bytes_per_step": int(n_done * 12),
                       "steps": len(e2e_times), "wall_s_per_step": e2e_s,
                       "what": "mbpe_train_sharded(deduplicated corpus in host memory): every rank uploads its shard, sharded "
                               "merge loop, D2H merges (h2d bytes are per rank)"}
        # for the record: N independent replicas of the single-GPU trainer (the round-1 'value'; weak scaling, no exchange)
        trainer = pkg.Trainer(tok, off, w, device=local_rank)
        rep_ms, (rm, _, _) = timed_steps(lambda: trainer.run(a.vocab, a.mode, a.engine, stream), 1, 1)
        line["train"]["replicas"] = {"aggregate_merges_per_sec": world * len(rm) / (rep_ms / 1e3), "ms_per_run": rep_ms,
                                     "equals_sharded_merges": all_true(hashlib.sha256(rm.tobytes()).hexdigest() == model_sha),
                                     "what": "N independent replicas of mbpe_trainer_run on the same corpus (not a scaling number)"}
        trainer.close()

    # ---------------- parity at the FULL workload size: the CPU oracle trains the same deduplicated corpus ------------
    if not a.no_check and rank == 0:
        from oracle import oracle as O
        t0 = time.time()
        om, oc = O.train(tok, off, w, a.vocab, a.mode)
        line["train"]["oracle_check"] = {"merges_equal": bool(om.shape == merges.shape and (om == merges).all()),
                                         "counts_equal": bool(oc.shape == counts.shape and (oc == counts).all()),
                                         "oracle_s": time.time() - t0, "oracle": "oracle_train_indexed, 1 thread"}

    # ---------------- the other tie-break mode (the reference CLI's default is `first`) --------------------------------
    if not a.skip_first:
        other = "first" if a.mode == "lexical" else "lexical"
        if world == 1:
            o_ms, (o_m, o_c, o_st) = timed_steps(lambda: trainer.run(a.vocab, other, a.engine, stream), 1, a.steps)
        else:
            o_ms, (o_m, o_c, o_st) = timed_steps(lambda: strainer.run(a.vocab, other, stream), 1, a.steps)
        dumps.update({f"train_{other}_merges": o_m, f"train_{other}_counts": o_c})
        leg = {"mode": other, "value": len(o_m) / (o_ms / 1e3), "unit": "merges/s", "ms_per_step": o_ms, "merges": int(len(o_m)),
               "merges_sha256": hashlib.sha256(o_m.tobytes()).hexdigest()}
        if not a.no_check and rank == 0:
            from oracle import oracle as O
            t0 = time.time()
            om, oc = O.train(tok, off, w, a.vocab, other)
            leg["oracle_check"] = {"merges_equal": bool(om.shape == o_m.shape and (om == o_m).all()),
                                   "counts_equal": bool(oc.shape == o_c.shape and (oc == o_c).all()), "oracle_s": time.time() - t0}
        line["train_" + other] = leg
        line["gpu_launches"] += int(o_st["n_launches"]) * a.steps
    if world == 1:
        trainer.close()
    else:
        strainer.close()

    # ---------------- encode: BASELINE config 4 ------------------------------------------------------------------------
    if not a.skip_encode:
        # The whole job: --encode-gib of text = the synthetic encode corpus, generated in 1 MiB blocks that end on a
        # newline, so every block boundary is a chunk boundary. mbpe_plan_shards cuts that list into `world` contiguous
        # byte-balanced ranges; rank r holds its range resident in batches of --encode-batch-mib.
        n_blocks = int(a.encode_gib * 1024)
        plan = pkg.plan_shards(np.arange(n_blocks + 1, dtype=np.uint64) * MIB, world)
        blk0, blk1 = int(plan[rank]), int(plan[rank + 1])
        pt = pkg.Pretok(device=local_rank)
        batches, t_egen, t_esplit = [], 0.0, 0.0
        for b0 in range(blk0, blk1, a.encode_batch_mib):
            nb = min(a.encode_batch_mib, blk1 - b0) * MIB
            t0 = time.time()
            etext = pkg.synth_corpus(SEED_ENCODE, nb, first_block=b0)
            t_egen += time.time() - t0
            d_bytes = torch.from_numpy(etext).to(dev)
            d_off_full = torch.empty(nb + 2, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            t0 = time.time()
            nck = pt.split_device(d_bytes.data_ptr(), nb, d_off_full.data_ptr(), nb + 2)  # device matcher
            t_esplit += time.time() - t0
            d_off = d_off_full[:nck + 1].clone()
            del d_off_full
            batches.append({"first_block": b0, "n_bytes": nb, "n_chunks": nck, "d_bytes": d_bytes, "d_off": d_off, "n_ids": 0})
        cap_ids = max(bt["n_bytes"] for bt in batches)
        d_out = torch.empty(cap_ids, dtype=torch.int32, device=dev)
        d_n = torch.zeros(1, dtype=torch.int64, device=dev)
        my_bytes = sum(bt["n_bytes"] for bt in batches)
        my_chunks = sum(bt["n_chunks"] for bt in batches)

        def encode_pass(enc):
            for bt in batches:
                enc.encode_device(bt["d_bytes"].data_ptr(), bt["n_bytes"], bt["d_off"].data_ptr(), bt["n_chunks"],
                                  d_out.data_ptr(), cap_ids, d_n.data_ptr(), stream)

        # cold steps: every step starts with a FRESH encoder (empty caches), created outside the timed region
        n_warm, n_steps = max(1, min(a.warmup, 3)), max(1, a.steps)
        encs = []
        for _ in range(n_warm + n_steps):
            e = pkg.Encoder(merges, device=local_rank)
            e.reserve(cap_ids, max(bt["n_chunks"] for bt in batches))
            encs.append(e)
        it = iter(encs)
        cold_ms, _ = timed_steps(lambda: encode_pass(next(it)), n_warm, n_steps)
        enc = encs[-1]
        launches_cold = enc.launches()
        for e in encs[:-1]:
            e.close()
        # the same text again through the now-warm caches, for the record (not the headline: config 4 sees its text once)
        warm_ms, _ = timed_steps(lambda: encode_pass(enc), 1, n_steps)
        if a.dump_outputs and rank == 0:  # the last timed step left the ids of the last batch in d_out
            dumps["encode_ids"] = d_out[torch.from_numpy(dump_rows(int(d_n.item()))).to(dev)].cpu().numpy().view(np.uint32)
        # untimed: id counts of every batch for the algorithmic-byte figure; the first batch's ids are kept for the checks
        first_ids = None
        for bt in reversed(batches):
            enc.encode_device(bt["d_bytes"].data_ptr(), bt["n_bytes"], bt["d_off"].data_ptr(), bt["n_chunks"],
                              d_out.data_ptr(), cap_ids, d_n.data_ptr(), stream)
            bt["n_ids"] = int(d_n.item())
        my_ids = sum(bt["n_ids"] for bt in batches)
        tot_bytes, tot_chunks, tot_ids = (int(sum_over_ranks(x)) for x in (my_bytes, my_chunks, my_ids))
        b_enc = tot_bytes + 4 * tot_chunks + 4 * tot_ids  # SURVEY 8(d)
        bt0 = batches[0]  # its ids are in d_out now
        # size-independent property on the device at full batch size: decode(encode(x)) == x
        d_txt = torch.empty(bt0["n_bytes"] + 64, dtype=torch.uint8, device=dev)
        d_ntxt = torch.zeros(1, dtype=torch.int64, device=dev)
        dec_ms, _ = timed_steps(lambda: enc.decode_device(d_out.data_ptr(), bt0["n_ids"], d_txt.data_ptr(), bt0["n_bytes"] + 64,
                                                          d_ntxt.data_ptr(), stream), max(1, min(a.warmup, 3)), n_steps)
        n_txt = int(d_ntxt.item())
        if a.dump_outputs and rank == 0:
            dumps["decode_bytes"] = d_txt[torch.from_numpy(dump_rows(n_txt)).to(dev)].cpu().numpy()
        roundtrip = all_true(n_txt == bt0["n_bytes"] and bool(torch.equal(d_txt[:n_txt], bt0["d_bytes"])))
        b_dec = int(sum_over_ranks(4 * bt0["n_ids"] + n_txt))
        dec_bytes = int(sum_over_ranks(n_txt))
        trd = ncu_traffic("k_decode_lean")
        line["decode"] = {
            "metric": "bpe_decode_mb_per_sec", "value": dec_bytes / 1e6 / (dec_ms / 1e3), "unit": "MB/s", "ms_per_step": dec_ms,
            "n_ids": int(sum_over_ranks(bt0["n_ids"])), "bytes_out": dec_bytes, "equals_input_text": roundtrip,
            "roofline": {"bound": "hbm", "achieved": b_dec / 1e9 / (dec_ms / 1e3), "peak": peak * world, "unit": "GB/s",
                         "frac": b_dec / 1e9 / (dec_ms / 1e3) / (peak * world), "traffic": trd["dram_bytes_per_launch"] if trd else None,
                         "traffic_detail": trd, "peak_source": peak_src, "kernel": "k_decode_lean",
                         "algorithmic_bytes_per_step": b_dec},
        }
        first_ids_host = d_out[:bt0["n_ids"]].cpu().numpy().view(np.uint32) if rank == 0 else None
        # e2e: host text in, host ids out through the Tokenizer mirror (H2D + device split + merge scan + D2H), the same
        # batches, text and ids in pinned host memory; a FRESH tokenizer (cold caches) sees every batch once
        model_file = os.path.join(tempfile.gettempdir(), f"bench_{os.getpid()}_{rank}.model")
        pkg.write_model(model_file, gpt4, None, merges)
        text_pinned_e = torch.empty(cap_ids, dtype=torch.uint8, pin_memory=True)
        ids_pinned = torch.empty(cap_ids, dtype=torch.int32, pin_memory=True)
        ids_out = ids_pinned.numpy().view(np.uint32)
        tke = pkg.Tokenizer(gpt4, device=local_rank)
        tke.load(model_file)
        warm_txt = pkg.synth_corpus(SEED_ENCODE + 7, 64 * MIB)
        text_pinned_e.numpy()[:len(warm_txt)] = warm_txt
        tke.encode(text_pinned_e.numpy()[:len(warm_txt)], out=ids_out)  # builds the device tables and pipeline buffers (untimed)
        tke.close()
        tke = pkg.Tokenizer(gpt4, device=local_rank)
        tke.load(model_file)
        tke.encode(text_pinned_e.numpy()[:MIB], out=ids_out)  # device tables of the fresh tokenizer; its caches have seen 1 MiB
        e2e_enc_s, e2e_ids = 0.0, 0
        barrier()
        for bt in batches:
            text_pinned_e.numpy()[:bt["n_bytes"]] = bt["d_bytes"].cpu().numpy()  # (untimed: refills the pinned input buffer)
            t0 = time.time()
            ids = tke.encode(text_pinned_e.numpy()[:bt["n_bytes"]], out=ids_out)
            e2e_enc_s += time.time() - t0
            e2e_ids += len(ids)
            if bt is batches[0] and rank == 0:
                assert np.array_equal(ids, first_ids_host), "Tokenizer::encode and mbpe_encode_device disagree"
        e2e_enc_s = max_over_ranks(e2e_enc_s)
        # the hot-path boundary alone: mbpe_encode(host bytes + host u64 chunk offsets), one batch
        e2e_abi = None
        if rank == 0:
            nb_abi = min(bt0["n_bytes"], 256 * MIB)
            etb = bt0["d_bytes"][:nb_abi].cpu().numpy().tobytes()
            off_abi = bt0["d_off"].cpu().numpy().view(np.uint32).astype(np.uint64)
            n_abi = int(np.searchsorted(off_abi, nb_abi, side="right")) - 1
            while off_abi[n_abi] != nb_abi and n_abi > 0:  # (block boundaries are chunk boundaries: exact hit expected)
                n_abi -= 1
            etb = etb[:int(off_abi[n_abi])]
            out_abi = np.ones(len(etb), np.uint32)  # caller-owned, already touched: the timed call pays no page faults for it
            off_abi = np.ascontiguousarray(off_abi[:n_abi + 1])
            enc.encode(etb, off_abi, out=out_abi)  # first call: sizes the handle's pinned staging buffers (untimed)
            t0 = time.time()
            ids_abi = enc.encode(etb, off_abi, out=out_abi)
            abi_s = time.time() - t0
            e2e_abi = {"value": len(etb) / 1e6 / abi_s, "unit": "MB/s", "bytes": len(etb),
                       "equals_device_path": bool(np.array_equal(ids_abi, first_ids_host[:len(ids_abi)])),
                       "what": "mbpe_encode(pageable host bytes + host u64 chunk offsets): staging + H2D + merge scan + D2H"}
        tre = ncu_traffic("k_encode_tiles")
        line["encode"] = {
            "metric": "bpe_encode_mb_per_sec", "value": tot_bytes / 1e6 / (cold_ms / 1e3), "unit": "MB/s",
            "ms_per_step": cold_ms, "ms_per_gib": cold_ms / (tot_bytes / world / 2**30), "bytes_per_step": tot_bytes,
            "n_chunks": tot_chunks, "n_tokens": tot_ids, "scaling": "strong",
            "workload": f"BASELINE config 4: encode {a.encode_gib} GiB of DISTINCT synthetic text (seed 0x{SEED_ENCODE:X}) with the "
                        f"{a.vocab}-vocab model just trained, streamed once through caches that start EMPTY; contiguous ranges of "
                        f"whole chunks per rank (mbpe_plan_shards), text / boundaries / ids resident in HBM, every batch >> L2",
            "warm_caches": {"ms_per_step": warm_ms, "value": tot_bytes / 1e6 / (warm_ms / 1e3),
                            "frac": b_enc / 1e9 / (warm_ms / 1e3) / (peak * world),
                            "what": "the same text a second time through the same encoder (caches warm) -- not the headline"},
            "roofline": {"bound": "hbm", "achieved": b_enc / 1e9 / (cold_ms / 1e3), "peak": peak * world, "unit": "GB/s",
                         "frac": b_enc / 1e9 / (cold_ms / 1e3) / (peak * world), "traffic": tre["dram_bytes_per_launch"] if tre else None,
                         "traffic_detail": tre, "peak_source": peak_src + (f" x {world} GPUs" if world > 1 else ""),
                         "kernel": "k_encode_tiles", "algorithmic_bytes_per_step": int(b_enc)},
            "e2e": {"value": tot_bytes / 1e6 / e2e_enc_s, "unit": "MB/s", "h2d_bytes_per_step": int(tot_bytes),
                    "d2h_bytes_per_step": int(4 * sum_over_ranks(e2e_ids)), "wall_s": e2e_enc_s,
                    "what": "mbpe_tokenizer_encode(text) = Tokenizer::encode per batch, text and ids in pinned host memory, fresh "
                            "tokenizer: H2D text + device split + merge scan + D2H ids; sum of the per-batch call times, max over ranks"},
            "e2e_abi": e2e_abi,
            "host_generate_s": t_egen, "device_split_s": t_esplit, "roundtrip_ok": roundtrip,
            "gpu_launches": int(launches_cold),
        }
        line["gpu_launches"] += int(launches_cold) * n_steps + n_steps
        os.unlink(model_file)

    # ---------------- config 5: 8 GiB, vocab 100000, text sharded over the ranks ---------------------------------------
    if a.config5 or world == 8:
        blocks = a.config5_gib * 1024
        plan5 = pkg.plan_shards(np.arange(blocks + 1, dtype=np.uint64) * MIB, world)
        b0, b1 = int(plan5[rank]), int(plan5[rank + 1])
        t0 = time.time()
        text5 = pkg.synth_corpus(SEED_CONFIG5, (b1 - b0) * MIB, first_block=b0)
        t_gen5 = time.time() - t0
        pin5 = torch.empty(len(text5), dtype=torch.uint8, pin_memory=True)
        pin5.numpy()[:] = text5
        del text5
        times5, err5 = [], None
        for i in range(2):  # first call sizes the resident buffers
            barrier()
            t0 = time.time()
            try:
                if world == 1:
                    tk.train(pin5.numpy(), a.config5_vocab, a.mode)
                    m5 = tk.merges()
                    st5 = tk.last_train_stats()
                else:
                    m5, c5, st5 = comm.train_text(pin5.numpy(), a.config5_vocab, a.mode)
            except Exception as ex:  # (the headline legs above must not be lost to this one)
                err5 = f"{type(ex).__name__}: {ex}"
            torch.cuda.synchronize()
            if not all_true(err5 is None):
                err5 = err5 or "failed on another rank"
                break
            barrier()
            times5.append(time.time() - t0)
        if err5 is not None:
            line["config5"] = {"error": err5}
            m5, st5, times5 = np.zeros((0, 2), np.uint32), {}, [float("nan")]
        s5 = max_over_ranks(times5[-1])
        leg5 = {"workload": f"BASELINE config 5: train {a.config5_gib} GiB synthetic corpus (seed 0x{SEED_CONFIG5:X}), --vocab-size "
                            f"{a.config5_vocab} gpt4 -c {a.mode}, text sharded over {world} GPU(s) in pinned host memory",
                "value": len(m5) / s5, "unit": "merges/s", "wall_s_text_to_model": s5, "merges": int(len(m5)),
                "merges_sha256": hashlib.sha256(m5.tobytes()).hexdigest(), "gpu_ms_merge_loop": st5.get("gpu_ms"),
                "host_generate_s": t_gen5,
                "what": "Tokenizer::train(text)" if world == 1 else
                        "mbpe_train_text_sharded: every rank splits + deduplicates ITS part of the text on its GPU, one all-gather of "
                        "the unique chunks, merge loop on the combined corpus"}
        if world > 1:
            h = torch.tensor(list(hashlib.sha256(m5.tobytes()).digest()), dtype=torch.int32, device=dev)
            h0 = h.clone()
            dist.broadcast(h0, 0)
            leg5["same_merges_on_every_rank"] = all_true(bool((h == h0).all()))
        if err5 is None:
            line["config5"] = leg5
            dumps["config5_merges"] = m5
        del pin5

    # ---------------- CPU baseline (rank 0, N == 1 only): the compiled reference on bounded samples --------------------
    if rank == 0 and world == 1 and not a.skip_cpu_baseline:
        cb, ref_merges, sample = ref_train_sample(a.ref_sample_mib, a.ref_merges, a.mode, a.corpus_mib * MIB)
        # parity on the same sample: our merge list for that slice must equal the reference's
        ss, se = pkg.split(gpt4, sample)
        st_, so_, sw_ = pkg.dedup(sample, ss, se)
        sm_, _, _ = pkg.train(st_, so_, sw_, 256 + a.ref_merges, a.mode, a.engine)
        cb["gpu_equals_reference_on_sample"] = bool(sm_.shape == ref_merges.shape and (sm_ == ref_merges).all())
        cb["reference_full_16MiB_run"] = reference_full_run_record()
        line["cpu_baseline"] = cb
        if not a.skip_encode:
            with tempfile.TemporaryDirectory() as td:
                mp = os.path.join(td, "bench.model")
                pkg.write_model(mp, gpt4, None, merges)
                ecb, sample_text = ref_encode_sample(mp, a.ref_encode_mib)
            # the reference's id stream for that slice must be the head of ours (the slice ends at a regex-safe cut)
            n_ref = ecb["n_ids"]
            ecb["gpu_equals_reference_on_sample"] = bool(
                n_ref <= len(first_ids_host) and hashlib.sha256(first_ids_host[:n_ref].tobytes()).hexdigest() == ecb["sha256"])
            line["encode"]["cpu_baseline"] = ecb

    tk.close()
    if comm:
        comm.close()
    if clocks:
        line["clocks"] = clocks.summary()
    if rank == 0:
        if a.dump_outputs:
            write_outputs(a.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
