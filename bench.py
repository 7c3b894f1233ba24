#!/usr/bin/env python3
"""bench.py — messages/sec through the hot path (parse -> link-extract -> filter/dedup -> JSONL).

Usage:
    python bench.py [--config {2,3,4,5}] --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

--config selects the BASELINE.json workload (default 2 = configs[1], the configuration the metric is quoted on):
  2  10 M synthetic Telegram mixed text/photo/video-metadata messages per GPU, parse + link-extract + dedup + JSONL
  3  100 M Telegram text messages per GPU, t.me/@username link-extract + hash-dedup snowball frontier (no JSONL)
  4  50 M synthetic YouTube video-metadata records per GPU, parse + JSONL, streamed in resident-sized batches
  5  1 B-message snowball sharded over the ranks (1e9 / N messages per GPU), NCCL set merge, frontier capacity 2^25
N > 1 is weak scaling for configs 2-4 (every rank takes its own shard of the same generator: record-index
sharding, no data-path collective) and strong scaling for config 5; the ranks merge their dedup sets once per step.

  * value  = whole-job records/s with the packed batches already resident in HBM (kernels only).
  * e2e    = the same metric through the public C ABI with HOST buffers: host -> device copy of every input array
    and device -> pinned-host copy of the results (JSONL blob, line offsets, status, per-record links) inside the
    timed region, pipelined over the library's three staging slots.
  * roofline: the dominant kernel of the workload — algorithmic bytes per launch / its CUDA-event duration measured
    live on the launching stream, against MEASURED_PEAKS.json; plus the whole-step figure (SURVEY.md §8d bytes).
  * cpu_baseline / --impl reference: the CPU oracle (C restatement of the reference's Go path — the reference itself
    cannot be built here, there is no Go toolchain) on the box's host cores, same run flags, same corpus.
  * --dump-outputs DIR: what the last timed resident step handed its caller, as .npy files (OutputDump): per run the
    result counts and seeded 4 KB windows of the JSONL, then a seeded sample of the dedup set's keys.
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "messages/sec parsed+link-extracted+JSONL"
UNIT = "messages/s"
E2E_CHUNK = int(os.environ.get("TGI_BENCH_CHUNK", 500_000))   # records per C-ABI call in the e2e leg
SLOT_MAX = int(os.environ.get("TGI_BENCH_SLOT_MAX", 42_000_000))  # records per resident slot (links-only configs)
GEN_BUDGET_S = float(os.environ.get("TGI_BENCH_GEN_BUDGET_S", 300))  # host time the synthetic-corpus generator may take per rank
ORC_RUN_SLICES, ORC_RUN_PIN = 0x10000, 0x20000

J, L, F, S = 0x01, 0x02, 0x04, 0x10  # TGI_RUN_JSONL / LINKS / FRONTIER / SKIP_SELF

# --dump-outputs: the JSONL and the dedup set of a step are gigabytes, so a fixed, seeded sample of them is written
# (byte values as float32: at most 43 MB whatever the number of resident runs, small enough to keep beside each build)
DUMP_SEED = 0x5EED0D0
DUMP_WINDOW = 4096               # JSONL bytes per sampled window
DUMP_JSONL_BYTES = 6 << 20       # JSONL bytes sampled over the step, split evenly over its resident runs
DUMP_FRONTIER_ROWS = 1 << 17     # dedup-set keys sampled (32 bytes each)


def configs():
    env = lambda k, d: int(os.environ.get(k, d))
    return {
        2: dict(kind="tg", profile=2, seed=0x5EED0002, n=env("TGI_BENCH_N", 10_000_000), flags=J | L | F | S, scaling="weak",
                cpu_n=env("TGI_BENCH_CPU_SAMPLE", 2_000_000), ref_n=env("TGI_BENCH_REF_N", 10_000_000), e2e_n=None,
                fcap=1 << 23,
                workload="configs[1]: 10M synthetic Telegram mixed text/photo/video-metadata messages, parse+link-extract+dedup+JSONL"),
        3: dict(kind="tg", profile=3, seed=0x5EED0003, n=env("TGI_BENCH_N", 100_000_000), flags=L | F | S, scaling="weak",
                cpu_n=env("TGI_BENCH_CPU_SAMPLE", 5_000_000), ref_n=env("TGI_BENCH_REF_N", 20_000_000),
                e2e_n=env("TGI_BENCH_E2E_N", 20_000_000), fcap=1 << 25,
                workload="configs[2]: 100M-message t.me/@username link-extract + hash-dedup snowball frontier"),
        4: dict(kind="yt", profile=0, seed=0x5EED0004, n=env("TGI_BENCH_N", 50_000_000), flags=J | L | F, scaling="weak",
                cpu_n=env("TGI_BENCH_CPU_SAMPLE", 1_000_000), ref_n=env("TGI_BENCH_REF_N", 2_000_000),
                e2e_n=env("TGI_BENCH_E2E_N", 5_000_000), fcap=1 << 23, batch=env("TGI_BENCH_YT_BATCH", 5_000_000),
                workload="configs[3]: 50M synthetic YouTube video-metadata records, parse+JSONL"),
        5: dict(kind="tg", profile=3, seed=0x5EED0005, n=env("TGI_BENCH_N", 1_000_000_000), flags=L | F | S, scaling="strong",
                cpu_n=env("TGI_BENCH_CPU_SAMPLE", 5_000_000), ref_n=env("TGI_BENCH_REF_N", 20_000_000),
                e2e_n=env("TGI_BENCH_E2E_N", 20_000_000), fcap=1 << 25,
                workload="configs[4]: 1B-message snowball: parse+extract+global hash-dedup sharded across the ranks with NCCL set-merge"),
    }


def ensure_built():
    import __graft_entry__ as g
    need = [os.path.join(ROOT, "distributed_crawler_b200", "libtgingest.so"),
            os.path.join(ROOT, "corpus", "libtgcorpus.so"), os.path.join(ROOT, "oracle", "libtgoracle.so")]
    if not all(os.path.exists(p) for p in need):
        g.build()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.p = gpu_index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def bind_numa(local_rank: int):
    """Keep this rank's threads (and so its pinned staging pages) on the NUMA node of its GPU."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        for line in out.splitlines():
            f = line.split()
            if f and f[0] == f"GPU{local_rank}":
                # columns: GPU0.. NICs.. "CPU Affinity" "NUMA Affinity" ...: take the first a-b[,c-d] token
                for tok in f[1:]:
                    if tok and tok[0].isdigit() and ("-" in tok or "," in tok):
                        cpus = set()
                        for part in tok.split(","):
                            a, _, b = part.partition("-")
                            cpus.update(range(int(a), int(b or a) + 1))
                        os.sched_setaffinity(0, cpus)
                        return tok
    except Exception:
        pass
    return None


def host_cpus() -> tuple[int, str]:
    """CPUs this process may really use: the cgroup CPU quota (cpu.max) caps what os.cpu_count() advertises —
    more runnable threads than the quota only get throttled."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    why = f"{n} schedulable CPUs"
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            q = max(1, int(int(quota) / int(period)))
            if q < n:
                n, why = q, f"cgroup cpu.max {quota}/{period} = {q} CPUs (of {len(os.sched_getaffinity(0))} visible)"
    except (OSError, ValueError):
        pass
    return n, why


def stratified(n_items: int, k: int, rng) -> "np.ndarray":
    """k sorted indices in [0, n_items): one uniformly drawn index in each of k equal strata (all of them if k >= n_items)"""
    import numpy as np
    if k >= n_items:
        return np.arange(n_items, dtype=np.int64)
    return np.minimum((np.arange(k) + rng.random(k)) * (n_items / k), n_items - 1).astype(np.int64)


class OutputDump:
    """What the timed path hands its caller in one step, for --dump-outputs.  Per resident run: the result counts and
    seeded windows of the JSONL the run left on the device; after the step: a seeded sample of the dedup set's keys
    (the merged global set when the ranks merge).  Same arguments -> same corpus -> same windows and rows, so two
    builds can be compared file by file."""

    def __init__(self, eng, n_runs: int):
        import numpy as np
        self.eng, self.np = eng, np
        self.windows_per_run = max(1, DUMP_JSONL_BYTES // DUMP_WINDOW // n_runs)
        self.counts, self.at, self.windows = [], [], []

    def run(self, slot, r):
        """sample run r right after it returned, before the next run reuses its slot"""
        np = self.np
        k = len(self.counts)
        self.counts.append([r.n, r.jsonl_len, r.n_links, r.n_new, r.frontier_size])
        if not r.jsonl_len:
            return
        w = min(DUMP_WINDOW, r.jsonl_len)
        rng = np.random.default_rng([DUMP_SEED, k])
        for off in stratified(r.jsonl_len - w + 1, self.windows_per_run, rng):
            row = np.full(DUMP_WINDOW, -1.0, np.float32)  # -1: past the end of a JSONL shorter than one window
            row[:w] = np.frombuffer(self.eng.read_jsonl(slot, int(off), w), np.uint8)
            self.windows.append(row)
            self.at.append([k, off])

    def write(self, out_dir: str, keys):
        """keys: the (n, 32) uint8 dedup set after the step"""
        np = self.np
        rows = stratified(len(keys), DUMP_FRONTIER_ROWS, np.random.default_rng([DUMP_SEED, 1 << 20]))
        arrays = {
            "run_counts": np.array(self.counts, np.float64).reshape(-1, 5),  # n, jsonl_len, n_links, n_new, frontier_size
            "jsonl_window_at": np.array(self.at, np.float64).reshape(-1, 2),  # run, byte offset of the window
            "jsonl_windows": np.array(self.windows, np.float32).reshape(-1, DUMP_WINDOW),
            "frontier_rows": rows.astype(np.float64),
            "frontier_keys": keys[rows].astype(np.float32),
        }
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)
        return sum(a.nbytes for a in arrays.values())


def make_corpus(cfg, n, first, threads):
    from distributed_crawler_b200.corpus import Corpus, YtCorpus
    if cfg["kind"] == "yt":
        return YtCorpus(n, seed=cfg["seed"], first=first, nthreads=threads)
    return Corpus(n, seed=cfg["seed"], first=first, profile=cfg["profile"], nthreads=threads)


def orc_run(o, cfg, batch, flags, nthreads):
    return (o.youtube if cfg["kind"] == "yt" else o.telegram)(batch, flags, nthreads=nthreads, copy=False)


def cpu_baseline(cfg, batch, cores):
    """The oracle on the host cores, same run flags: all cores, and one thread on a twentieth of the sample."""
    from oracle import pyoracle
    from oracle.pyoracle import Oracle
    flags = cfg["flags"] | ORC_RUN_SLICES | ORC_RUN_PIN
    o = Oracle()
    orc_run(o, cfg, batch, flags, cores)  # warm-up: grow the context-owned buffers
    dt = None
    for _ in range(3):  # best of three: the sample is short and the box's other tenants show up in a single run
        pyoracle.lib().orc_frontier_clear(o.h)
        t0 = time.perf_counter()
        orc_run(o, cfg, batch, flags, cores)
        d = time.perf_counter() - t0
        dt = d if dt is None else min(dt, d)
    o.close()
    o1 = Oracle()
    n1 = max(1, batch.n // 20)
    sub = batch.slice(0, n1) if hasattr(batch, "slice") else None
    v1 = None
    if sub is not None:
        orc_run(o1, cfg, sub, cfg["flags"], 1)
        pyoracle.lib().orc_frontier_clear(o1.h)
        t1 = time.perf_counter()
        orc_run(o1, cfg, sub, cfg["flags"], 1)
        v1 = n1 / (time.perf_counter() - t1)
    o1.close()
    return batch.n / dt, dt, v1


def run_reference(args, cfg, rank):
    """--impl reference: the reference path's CPU implementation (oracle port) on the host cores."""
    if rank != 0:
        return
    from oracle import pyoracle
    from oracle.pyoracle import Oracle
    cores, cores_why = host_cpus()
    n = min(cfg["ref_n"], cfg["n"])
    c = make_corpus(cfg, n, 0, min(cores, 64))
    flags = cfg["flags"] | ORC_RUN_SLICES | ORC_RUN_PIN
    o = Oracle()
    for _ in range(max(args.warmup, 1)):
        pyoracle.lib().orc_frontier_clear(o.h)
        orc_run(o, cfg, c.batch, flags, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pyoracle.lib().orc_frontier_clear(o.h)
        orc_run(o, cfg, c.batch, flags, cores)
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    # one thread, for the per-thread efficiency of the parallel arm
    v1 = None
    if hasattr(c.batch, "slice"):
        sub = c.batch.slice(0, max(1, n // 50))
        o1 = Oracle()
        orc_run(o1, cfg, sub, cfg["flags"], 1)
        pyoracle.lib().orc_frontier_clear(o1.h)
        t1 = time.perf_counter()
        orc_run(o1, cfg, sub, cfg["flags"], 1)
        v1 = sub.n / (time.perf_counter() - t1)
        o1.close()
    same = n == cfg["n"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": cfg["scaling"],
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": cfg["workload"], "bench_config": args.config, "run_flags": cfg["flags"],
                       "sample": ("the whole corpus" if same else f"first {n} records of the same seeded corpus") + " per step",
                       "same_corpus_as_gpu_arm": same},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "one_thread": v1, "per_thread_efficiency": (v / cores / v1) if v1 else None,
                             "cores_basis": cores_why,
                             "sample": f"{n} records x {args.steps} steps, C restatement of the Go path, {cores} threads pinned one per core, "
                                       "each worker keeps its own output (no global concatenation, like the reference's per-channel files), "
                                       "sharded frontier insert"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    def positive(s):
        v = int(s)
        if v < 1:
            raise argparse.ArgumentTypeError("must be at least 1")
        return v

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive, default=5, help="timed steps of the resident leg and of the host-buffer leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of what the last resident step computed as "
                         "DIR/<name>.npy; the corpus is then never cut to the generator's time budget")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    cfg = configs()[args.config]
    ensure_built() if rank == 0 or world == 1 else time.sleep(0)
    if args.impl == "reference":
        run_reference(args, cfg, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from distributed_crawler_b200 import abi
    from distributed_crawler_b200.engine import Engine

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    numa = bind_numa(local)  # pinned result / staging pages on the GPU's own NUMA node, also at N = 1
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner to stdout when the first communicator is created; the bench contract
        # is ONE JSON line there, so stdout points at stderr until the communicator exists
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            t = torch.zeros(1, device=dev)
            dist.all_reduce(t)
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    cores, cores_why = host_cpus()
    gen_threads = max(1, min((os.cpu_count() or 1) // max(world, 1), 64))
    is_yt = cfg["kind"] == "yt"
    RUN = cfg["flags"]
    want_json = bool(RUN & J)
    n = cfg["n"] // world if cfg["scaling"] == "strong" else cfg["n"]   # records per GPU
    n_asked = n
    # the corpus is generated on the host: keep that inside a time budget, whatever CPUs this box grants; a dump must
    # see the same corpus on every run, so it takes the configured size
    if n > 4_000_000 and not args.dump_outputs:
        t_probe = time.perf_counter()
        make_corpus(cfg, 1_000_000, rank * n, gen_threads).close()
        rate = 1_000_000 / (time.perf_counter() - t_probe)
        fit = int(rate * GEN_BUDGET_S)
        if world > 1:
            fit_t = torch.tensor([fit], dtype=torch.int64, device=dev)
            dist.all_reduce(fit_t, op=dist.ReduceOp.MIN)
            fit = int(fit_t.item())
        if fit < n:
            n = max(1_000_000, fit // 1_000_000 * 1_000_000)
    first = rank * n
    eng = Engine(device=local, frontier_capacity=cfg["fcap"])
    merger = None
    if world > 1:
        from distributed_crawler_b200.frontier_merge import make_merger
        merger = make_merger(eng, dev)

    # ---- resident batches: up to three slots for Telegram; YouTube streams `batch`-sized uploads through slot 0 ----
    t_gen = time.perf_counter()
    if is_yt:
        per = min(cfg["batch"], n)
        parts = [(a, min(a + per, n)) for a in range(0, n, per)]
    else:
        k = max(1, -(-n // SLOT_MAX)) if not want_json else 1
        if k > abi.SLOTS:
            raise SystemExit(f"{n} records per GPU need more than {abi.SLOTS} resident slots of {SLOT_MAX}")
        parts = [(n * i // k, n * (i + 1) // k) for i in range(k)]
    corpora = [make_corpus(cfg, b - a, first + a, gen_threads) for a, b in parts]
    in_bytes = sum(c.batch.input_bytes() for c in corpora)
    if not is_yt:
        for i, c in enumerate(corpora):
            eng.telegram_upload(i, c.batch)
    t_gen = time.perf_counter() - t_gen

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: kernels only, batches resident in HBM ------------------------------------------------
    class Acc:
        def __init__(self):
            self.launches = 0
            self.ms = {"kernel": 0.0, "parse": 0.0, "emit": 0.0, "main": 0.0, "frontier": 0.0}
            self.jsonl = self.links = self.lane_out = self.lane_in = 0
            self.upload_s = self.dump_s = 0.0

        def add(self, r):
            self.launches += r.gpu_launches
            for k2, v in (("kernel", r.kernel_ms), ("parse", r.parse_ms), ("emit", r.emit_ms), ("main", r.emit_main_ms),
                          ("frontier", getattr(r, "frontier_ms", 0.0))):
                self.ms[k2] += v
            self.jsonl += r.jsonl_len; self.links += r.n_links
            self.lane_out += r.main_bytes_out; self.lane_in += r.main_bytes_in

    def sample(acc, dump, slot, r):
        t_d = time.perf_counter()
        dump.run(slot, r)
        acc.dump_s += time.perf_counter() - t_d

    def step_resident(acc=None, dump=None):
        eng.frontier_clear()
        r = None
        if is_yt:
            for c in corpora:
                t_up = time.perf_counter()
                eng.youtube_upload(0, c.batch)
                if acc:
                    acc.upload_s += time.perf_counter() - t_up
                r = eng.youtube_run_resident(0, RUN | abi.RUN_NO_D2H)
                if acc:
                    acc.add(r)
                if dump:
                    sample(acc, dump, 0, r)
        else:
            for i in range(len(corpora)):
                r = eng.telegram_run_resident(i, RUN | abi.RUN_NO_D2H)
                if acc:
                    acc.add(r)
                if dump:
                    sample(acc, dump, i, r)
        gsize = r.frontier_size
        if merger:
            gsize = merger.merge()
        return gsize

    for _ in range(max(args.warmup, 3)):
        gsize = step_resident()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    acc = Acc()
    dump = OutputDump(eng, len(corpora)) if args.dump_outputs else None
    t0 = time.perf_counter()
    for i in range(args.steps):
        gsize = step_resident(acc, dump if i == args.steps - 1 else None)
    barrier()
    # YouTube: the uploads between resident batches are not part of `value`; nor is the sampling of --dump-outputs
    dt = time.perf_counter() - t0 - acc.upload_s - acc.dump_s
    clocks = sampler.stop()
    dump_bytes = None
    if dump:
        keys = merger.global_export() if merger else eng.frontier_export()  # the merged set's export is collective
        if rank == 0:
            dump_bytes = dump.write(args.dump_outputs, keys)
        del keys
    dt_t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt_t, op=dist.ReduceOp.MAX)
    dt_max = float(dt_t.item())
    value = n * world * args.steps / dt_max
    jsonl_len = acc.jsonl // args.steps
    n_links = acc.links // args.steps
    merge_stats = merger.stats() if merger else None

    # ---- e2e: host buffers through the C ABI, 3 slots pipelined ----------------------------------
    e2e = None
    if not args.no_e2e:
        e2e_n = min(cfg["e2e_n"] or n, n)
        if is_yt:
            subs = [make_corpus(cfg, min(E2E_CHUNK, e2e_n - a), first + a, gen_threads).batch for a in range(0, e2e_n, E2E_CHUNK)]
        else:
            subs, left = [], e2e_n
            for c in corpora:  # views copied once, outside the timed region
                m = min(left, c.batch.n)
                subs += [c.batch.slice(a, min(a + E2E_CHUNK, m)) for a in range(0, m, E2E_CHUNK)]
                left -= m
                if not left:
                    break
        staged = [eng.stage(s) for s in subs]  # library-owned pinned input staging (tgi_acquire_staging)
        submit = eng.youtube_submit if is_yt else eng.telegram_submit
        wait = eng.youtube_wait if is_yt else eng.telegram_wait

        def step_e2e():
            eng.frontier_clear()
            d2h = 0
            inflight = []
            for i, sub in enumerate(staged):
                slot = i % abi.SLOTS
                if len(inflight) == abi.SLOTS:
                    s0 = inflight.pop(0)
                    rr = wait(s0)
                    d2h += rr.d2h_bytes()
                    eng.release(s0)
                submit(slot, sub, RUN)
                inflight.append(slot)
            for s0 in inflight:
                rr = wait(s0)
                d2h += rr.d2h_bytes()
                eng.release(s0)
            if merger:
                merger.merge()
            return d2h

        for _ in range(2):
            d2h_bytes = step_e2e()
        barrier()
        e2e_steps = args.steps
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            d2h_bytes = step_e2e()
        barrier()
        dte = time.perf_counter() - t0
        dte_t = torch.tensor([dte], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dte_t, op=dist.ReduceOp.MAX)
        h2d_bytes = sum(s.input_bytes() for s in subs)
        e2e = {"value": e2e_n * world * e2e_steps / float(dte_t.item()), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": d2h_bytes, "steps": e2e_steps, "chunk_records": E2E_CHUNK, "slots": abi.SLOTS,
               "records_per_step_per_gpu": e2e_n, "input_staging": "tgi_acquire_staging (library-owned pinned memory)",
               "h2d_gbs_per_gpu": h2d_bytes * e2e_steps / dte / 1e9, "d2h_gbs_per_gpu": d2h_bytes * e2e_steps / dte / 1e9,
               "numa_cpus": numa}
        for s in staged:
            eng.unstage(s)
        del staged, subs

    # ---- page-sized calls: the granularity the reference calls ParseMessage / convertVideoToPost with ------------------
    page_calls = None
    if rank == 0 and not args.no_e2e and hasattr(corpora[0].batch, "slice"):
        import ctypes as C
        from distributed_crawler_b200.engine import lib
        call = lib().tgi_youtube_batch if is_yt else lib().tgi_telegram_batch
        page_calls = {"what": "blocking C-ABI call, host buffers in, host result out, mean of 100 calls after 5 warm-up calls; "
                              "same run flags as the step; one cooperative launch per call (csrc/tg_page.cuh, yt_page.cuh)"}
        for pn in ((50, 500) if is_yt else (100, 1000)):
            pb = corpora[0].batch.slice(0, pn)
            d = pb.descriptor()
            r = abi.ResultC()
            for i in range(105):
                if i == 5:
                    t0 = time.perf_counter()
                if call(eng.h, C.byref(d), RUN, C.byref(r)) != 0:
                    raise SystemExit("page call failed: " + lib().tgi_last_error(eng.h).decode())
                lib().tgi_result_release(eng.h, r.slot)
            page_calls[str(pn)] = {"ms_per_call": (time.perf_counter() - t0) / 100 * 1e3, "gpu_launches_per_call": int(r.gpu_launches),
                                   "result_bytes": int(r.jsonl_len)}

    if rank == 0:
        peak, peak_src = load_peaks()
        step_ms = dt_max / args.steps * 1e3
        per = lambda k2: acc.ms[k2] / args.steps
        traffic = load_traffic() or {}
        if want_json:
            # whole step (SURVEY.md §8d): every input byte read once, every output byte written once, 8 B line offset
            alg_bytes = in_bytes + jsonl_len + 8 * (n + 1)
            kname = "yt_emit_lane_kernel" if is_yt else "tg_emit_lane_kernel"
            # the main emit kernel (one lane per record): per record it reads the header (64 B), the line offset (8 B) and
            # the piece lengths of the size pass (32 B), writes the piece offsets (32 B), reads every source byte it copies
            # and writes the JSONL bytes it is responsible for; both sums are counted by the kernel itself
            # (tgi_result.main_bytes_in / main_bytes_out).  YouTube: the lane writer does not count: line bytes + inputs.
            k_alg = (acc.lane_out + acc.lane_in) // args.steps + n * (64 + 8 + 32 + 32) if not is_yt else in_bytes + jsonl_len
            k_ms = per("main")
        else:
            # link-extract + dedup (SURVEY.md §8d): mini header 24 B + text + entities + entity URLs read once,
            # 32 B key write + 64 B hash-slot read-modify-write per link reaching the set
            alg_bytes = sum(24 * c.batch.n + c.batch.strs.nbytes + c.batch.ents.nbytes + c.batch.aux.nbytes for c in corpora) + 96 * n_links
            kname = "tg_parse_kernel (+ tg_ent_map_kernel, tg_parse_ent_kernel)"
            k_alg = alg_bytes - 96 * n_links + 36 * n_links
            k_ms = per("parse")
        achieved = k_alg / (k_ms * 1e-3) / 1e9 if k_ms else 0.0
        roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic.get(kname + "_bytes_per_launch"),
                    "algorithmic_bytes_per_launch": k_alg, "kernel_ms": k_ms, "kernel_share_of_step": k_ms / step_ms,
                    "passes_ms": {"scan+size": per("parse"), "emit": per("emit"), "frontier": per("frontier"), "all_kernels": per("kernel")},
                    "step": {"algorithmic_bytes": alg_bytes, "achieved": alg_bytes / (step_ms * 1e-3) / 1e9,
                             "frac": alg_bytes / (step_ms * 1e-3) / 1e9 / peak}}
        cpu = None
        if not args.no_cpu:
            sample_n = min(cfg["cpu_n"], corpora[0].batch.n)
            sample = corpora[0].batch.slice(0, sample_n) if hasattr(corpora[0].batch, "slice") else make_corpus(cfg, sample_n, first, gen_threads).batch
            cpu_v, cpu_dt, cpu_v1 = cpu_baseline(cfg, sample, cores)
            cpu = {"value": cpu_v, "unit": UNIT, "cores": cores, "cores_basis": cores_why, "kind": "port", "one_thread": cpu_v1,
                   "per_thread_efficiency": (cpu_v / cores / cpu_v1) if cpu_v1 else None,
                   "sample": f"first {sample_n} records of the same corpus, {cpu_dt:.1f} s, C restatement of the Go path (oracle), same run flags, "
                             f"{cores} threads pinned one per core, warm, best of 3"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": cfg["workload"], "bench_config": args.config, "run_flags": RUN,
                       "records_per_gpu": n, "records_per_gpu_of_the_configuration": n_asked,
                       "reduced": (None if n == n_asked else f"the host generator (~{int(rate)} records/s on this rank's CPUs) would need more than "
                                                             f"{int(GEN_BUDGET_S)} s for {n_asked} records: TGI_BENCH_GEN_BUDGET_S"),
                       "resident_batches": len(corpora), "seed": hex(cfg["seed"]), "input_bytes_per_gpu": in_bytes,
                       "jsonl_bytes_per_gpu": jsonl_len, "links_per_gpu": n_links,
                       "l2": "inputs (%.1f GB) and outputs (%.1f GB) per step are far larger than the 126 MB L2" % (in_bytes / 1e9, jsonl_len / 1e9),
                       "timing": "wall clock around the K steps between barriers + synchronize, max over ranks"
                                 + ("; host->device uploads between the resident YouTube batches excluded" if is_yt else "")
                                 + ("; sampling of the last step's outputs excluded" if dump else ""),
                       "parallelism": f"record-index sharding x{world}" + ("; NCCL set merge per step: " + merger.describe() if merger else ""),
                       "frontier_unique": int(gsize), "corpus_gen_s": round(t_gen, 2)},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": acc.launches,
            "page_calls": page_calls,
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if merge_stats:
            line["merge"] = merge_stats
        if dump:
            line["dumped_outputs"] = {"dir": args.dump_outputs, "bytes": dump_bytes}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


if __name__ == "__main__":
    main()
