#!/usr/bin/env python3
"""bench.py -- input GB/s scanned by the double-array Aho-Corasick scan path on B200.

    python bench.py --gpus N --steps K --warmup W                    # headline: C3, find_overlapping_iter
    python bench.py --config {C3,C3-find,C2,C4,C5} ...               # the other BASELINE.json configs
    python bench.py --impl reference [--config ...] ...              # the reference's CPU path (C port)
    python bench.py ... --dump-outputs DIR                           # also write the last timed step's result

Headline workload (BASELINE.json configs[2] with the headline iterator): a bytewise automaton of 675 000
UniDic-like patterns; one *step* = one pass of find_overlapping_iter over a batch of 1 Mi haystacks x 4 KiB
(4 GiB of synthetic text) per GPU.  Weak scaling: every rank scans its own seeded shard and its placement
kernel stores the matches straight into rank 0's dense result buffer over NVLink peer memory (dach_group_*:
no collective); rank 0 ends every step holding the dense, rebased result of the whole N-GPU batch.
Steps are pipelined through two asynchronous jobs: the placement of step s runs beside the scan of step s+1;
all K placements complete inside the timed region.

`value` = device-resident throughput (inputs already in HBM), `e2e` = the same metric through the host-buffer
C-ABI call (pinned host -> device -> scan -> host, copies inside the timed region), `cpu_baseline` = the C port
of the crate's loops on the box's host cores, with an in-run parity check of the GPU result against it.
One JSON line is printed by rank 0.  See DESIGN.md section "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree, which may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

UNIT = "GB/s"

# name -> (synth config, crate iterator, automaton description, haystacks per step per GPU (None: the config's),
#          resident batches rotated through (inputs per pass must exceed L2), default steps)
CONFIGS = {
    "C3": dict(synth="C3", mode="find_overlapping_iter", what="675k-pat bytewise", batches=1, steps=20),
    "C3-find": dict(synth="C3", mode="find_iter", what="675k-pat bytewise", batches=1, steps=20),
    "C2": dict(synth="C2", mode="find_overlapping_iter", what="10k-pat ASCII bytewise", batches=4, steps=40),
    "C4": dict(synth="C4", mode="leftmost_find_iter", what="100k-pat CJK charwise LeftmostLongest", batches=1, steps=20),
    "C5": dict(synth="C5", mode="find_overlapping_iter", what="1M-pat bytewise, 12.5 GiB resident per GPU in 1 GiB windows",
               batches=13, steps=13, window=1024),
    # not a BASELINE.json config: C4's data on a bytewise LeftmostLongest automaton (the LmMachine kernel)
    "C4-bw": dict(synth="C4", mode="leftmost_find_iter", what="100k-pat CJK bytewise LeftmostLongest", batches=1, steps=20, variant="bytewise"),
}


def metric_name(cfg):
    return "input GB/s scanned, %s, %s" % (cfg["mode"], cfg["what"])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self, skip=0):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows[skip:] if len(self.rows) > skip else self.rows
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[2 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- workload --------------------------------------------------------------------------------------------

class Workload:
    """Patterns, text pool and window starts of one rank: everything is a pure function of (config, scale, rank)."""

    def __init__(self, name, scale, rank, pool_mib=None):
        from daachorse_b200 import synth as S

        self.S = S
        self.name = name
        self.spec = CONFIGS[name]
        self.cfg = S.config(self.spec["synth"], scale)
        self.mode_name = self.spec["mode"]
        self.ps = S.make_patterns(self.cfg)
        self.hay_len = self.cfg["hay_len"]
        self.n_total = self.cfg["n_haystacks"]               # haystacks resident per GPU
        self.window = min(self.spec.get("window") or self.n_total, self.n_total)  # haystacks per step
        if "window" not in self.spec:
            self.n_total = self.window * self.spec["batches"]
        nb = (pool_mib << 20) if pool_mib else self.cfg["pool_bytes"]
        self.pool, self.bounds = S.make_pool(self.cfg, self.ps, nb, seed=2 + 1000 * rank)
        self.starts = S.window_starts(self.bounds, len(self.pool), self.n_total, self.hay_len, seed=3 + 1000 * rank)
        self.charwise = self.spec.get("variant", self.cfg["variant"]) == "charwise"
        self.match_kind = self.cfg["match_kind"]

    def batch_ranges(self):
        """[lo, hi) haystack ranges of the batches a run rotates through."""
        if "window" in self.spec:  # C5: windows over the resident shard, the last one flush with its end
            out, lo = [], 0
            while lo + self.window <= self.n_total and len(out) < self.spec["batches"]:
                out.append((lo, lo + self.window))
                lo += self.window
            if len(out) < self.spec["batches"] and self.n_total > self.window and out[-1][1] < self.n_total:
                out.append((self.n_total - self.window, self.n_total))
            return out
        return [(k * self.window, (k + 1) * self.window) for k in range(self.spec["batches"])]

    def host_batch(self, lo, hi):
        """The same bytes the device batch holds, regenerated on the host (oracle side)."""
        text, offs = self.S.materialise_host(self.pool, self.starts[lo:hi], self.hay_len)
        if self.spec["synth"] == "C4":
            text = self.S.pad_to_char_boundary(text.reshape(hi - lo, self.hay_len)).reshape(-1)
        return text, offs

    def oracle(self):
        import oracle_api as O

        if self.charwise or self.match_kind:
            pats = [p.decode() for p in self.ps.as_list()] if self.charwise else self.ps.as_list()
            return O.OraclePma.build(pats, charwise=self.charwise, match_kind=self.match_kind)
        return O.OraclePma.build_packed(self.ps.blob, self.ps.offs)

    def automaton(self):
        import daachorse_b200 as D

        if self.charwise:
            return D.CharwiseDoubleArrayAhoCorasickBuilder.new().match_kind(self.match_kind).build(
                [p.decode() for p in self.ps.as_list()])
        return D.DoubleArrayAhoCorasickBuilder.new().match_kind(self.match_kind).build(self.ps.as_list())


def run_pipeline(steps, n_jobs, scan, place, finish):
    """The order in which a run issues its steps (callbacks take the step index; `finish` returns the step's total).
    With two jobs the scan of step s+1 is enqueued before step s is placed -- a shard group's place() blocks until
    the rank's host knows where its matches go (its own scan done, the lower ranks' counts published) -- and only
    after step s-1 has been finished, because it reuses that step's job."""
    tot = 0
    if steps <= 0:
        return tot
    scan(0)
    for s in range(steps):
        if n_jobs > 1:
            if s > 0:
                tot = finish(s - 1)      # step s-1 has landed: consume it ...
            if s + 1 < steps:
                scan(s + 1)              # ... its job scans step s+1 ...
            place(s)                     # ... while step s is exchanged
        else:
            place(s)
            tot = finish(s)
            if s + 1 < steps:
                scan(s + 1)
    if n_jobs > 1:
        tot = finish(steps - 1)
    return tot


def mode_ids(mode_name):
    import daachorse_b200 as D
    import oracle_api as O

    return {"find_iter": (D.FIND, O.FIND), "find_overlapping_iter": (D.FIND_OVERLAPPING, O.FIND_OVERLAPPING),
            "find_overlapping_no_suffix_iter": (D.FIND_OVERLAPPING_NO_SUFFIX, O.FIND_OVERLAPPING_NO_SUFFIX),
            "leftmost_find_iter": (D.LEFTMOST_FIND, O.LEFTMOST_FIND)}[mode_name]


DUMP_OFFSETS_MAX = 1 << 21       # offsets written (every k-th of them beyond that)
DUMP_TEXT_BYTES = 8 << 20        # haystack bytes in the sample whose matches are written ...
DUMP_HAYSTACKS_MAX = 1 << 16     # ... but no more haystacks than this
DUMP_MATCHES_MAX = 1 << 20       # and no more match rows than this
DUMP_SEED = 17


def dump_outputs(out_dir, matches, offsets, hay_len):
    """--dump-outputs: the result of one step as a caller receives it -- ``matches`` ((total, 3) int32 tensor of
    (start, end, value)) and ``offsets`` ((n + 1,) int64 tensor) -- written to out_dir as float64 .npy files, which
    hold every u32 position and value and every offset below 2**53 exactly.  At most about 41 MiB in all:

      offsets.npy          the offsets; every k-th of them (the first included) when there are more than 2**21
      match_haystacks.npy  a fixed, seeded sample of haystack indices (8 MiB of text, at most 65536 haystacks)
      match_counts.npy     the number of matches of each sampled haystack
      matches.npy          (m, 3): the sampled haystacks' matches in result order, their first 2**20 rows

    The sample depends on nothing but the number of haystacks and hay_len, so two builds run with the same
    arguments write arrays that can be compared element for element."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    o = offsets.cpu().numpy().astype(np.int64)
    n = o.size - 1
    stride = -(-o.size // DUMP_OFFSETS_MAX)
    k = min(n, DUMP_HAYSTACKS_MAX, max(1, DUMP_TEXT_BYTES // max(hay_len, 1)))
    hs = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=k, replace=False))
    lo, counts = o[hs], o[hs + 1] - o[hs]
    # row of every sampled match: haystack j's matches are rows lo[j] .. lo[j] + counts[j] - 1
    firsts = np.cumsum(counts) - counts
    rows = (np.repeat(lo - firsts, counts) + np.arange(int(counts.sum()), dtype=np.int64))[:DUMP_MATCHES_MAX]
    m = matches.index_select(0, torch.from_numpy(rows).to(matches.device)).cpu().numpy()
    arrays = {"offsets": o[::stride], "match_haystacks": hs, "match_counts": counts,
              "matches": m.view(np.uint32).reshape(-1, 3)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def cpu_sample(W, opma, omode, n_hay, min_seconds, threads):
    """Times orc_bench_batch on the first n_hay haystacks of the rank's first batch: repeated until min_seconds."""
    import oracle_api as O

    text, offs = W.host_batch(0, n_hay)
    O.bench_batch(opma, omode, text[: int(offs[min(n_hay, 64)])], offs[: min(n_hay, 64) + 1], threads)  # start the pool
    t0 = time.perf_counter()
    reps, total = 0, 0
    while True:
        total = O.bench_batch(opma, omode, text, offs, threads)
        reps += 1
        if time.perf_counter() - t0 >= min_seconds or reps >= 200:
            break
    dt = (time.perf_counter() - t0) / reps
    return text.size / dt / 1e9, dt, reps, total, text.size


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the path -- the C port in oracle/ (the Rust crate
    cannot be built in this image), on the crate's record layout, persistent pinned threads, bounded sample."""
    if rank != 0:
        return
    import oracle_api as O

    W = Workload(args.config, args.scale, 0, 32)
    _, omode = mode_ids(W.mode_name)
    opma = W.oracle()
    budget = O.cpu_budget()
    threads = budget["threads"]
    n_sample = min(W.window, max(threads * 4, args.ref_haystacks * 4096 // W.hay_len))  # about 1 GiB of the batch
    text, offs = W.host_batch(0, n_sample)
    for _ in range(max(args.warmup, 1)):
        O.bench_batch(opma, omode, text[: int(offs[min(n_sample, threads * 4)])], offs[: min(n_sample, threads * 4) + 1], threads)
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        total += O.bench_batch(opma, omode, text, offs, threads)
    dt = (time.perf_counter() - t0) / args.steps
    val = text.size / dt / 1e9
    one, _, _, _, _ = cpu_sample(W, opma, omode, min(n_sample, max(64, n_sample // max(threads, 1))), 1.0, 1)
    sample = "%d haystacks x %d B (%.1f MiB) of the %s batch per step" % (n_sample, W.hay_len, text.size / 2**20, args.config)
    line = {
        "impl": "reference", "metric": metric_name(W.spec), "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "%s: %s, %s, %d B haystacks" % (args.config, W.spec["what"], W.mode_name, W.hay_len),
                   "n_patterns": len(W.ps), "hay_len": W.hay_len, "matches_per_byte": total / args.steps / text.size},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "single_thread": one, "cpu": budget,
                         "note": "C restatement of daachorse 4.0.0's scan loops on the crate's array-of-structs records, "
                                 "-O3 -march=native built on this box, persistent pinned threads, matches stored to a "
                                 "per-thread ring (Rust toolchain unavailable: the crate itself cannot be built)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3", choices=sorted(CONFIGS))
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the config's batch (debug only)")
    ap.add_argument("--pool-mib", type=int, default=None)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--ref-haystacks", type=int, default=262144)
    ap.add_argument("--parity-frac", type=float, default=0.04, help="share of a batch checked against the oracle in the run")
    ap.add_argument("--option", action="append", default=[], help="kernel option name=value")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="one job, placement and next scan serialised (ablation)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR/*.npy (float64, a seeded sample; see dump_outputs)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = CONFIGS[args.config]["steps"]
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    import daachorse_b200 as D
    from daachorse_b200 import shard
    from daachorse_b200 import synth as S

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries exactly one JSON line: while the job runs, file descriptor 1 points at stderr, so that
    # anything a library writes to stdout (NCCL prints its version banner there under NCCL_DEBUG=VERSION)
    # lands in the log; the descriptor is restored just before rank 0 prints the line.
    saved_stdout = None
    try:
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
    except OSError:  # no usable stderr: leave stdout alone
        saved_stdout = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    t_setup = time.time()
    W = Workload(args.config, args.scale, rank, args.pool_mib)
    dmode, omode = mode_ids(W.mode_name)
    hay_len = W.hay_len
    pma = W.automaton()
    for kv in args.option:
        k, v = kv.split("=")
        pma.set_option(k, int(v))
    # ---- the rank's resident text: one gather on the device per batch ----
    pool_t = torch.from_numpy(W.pool).to(dev)
    starts_t = torch.from_numpy(W.starts).to(dev)
    ranges = W.batch_ranges()
    if "window" in W.spec:  # C5: the whole shard is resident, steps walk over it window by window
        text_all, offs_all = S.materialise_on_device(pool_t, starts_t, hay_len)
        batches = [(text_all[lo * hay_len: hi * hay_len], offs_all[: hi - lo + 1]) for lo, hi in ranges]
    else:
        batches = []
        for lo, hi in ranges:
            t, o = S.materialise_on_device(pool_t, starts_t[lo:hi], hay_len)
            if W.spec["synth"] == "C4":
                S.pad_to_char_boundary_device(t, hi - lo, hay_len)
            batches.append((t, o))
    del pool_t
    n = W.window                       # haystacks per step per GPU
    step_bytes = n * hay_len
    resident = sum(b[0].numel() for b in batches) if "window" not in W.spec else text_all.numel()
    torch.cuda.synchronize()

    # ---- sizing pass (not timed): match counts per batch, result buffers allocated once ----
    counts = []
    for t, o in batches:
        r = pma.scan_batch_device(dmode, t, o)
        counts.append(int(r.matches.shape[0]))
        del r
    cap_local = max(counts) + 4096
    if world > 1:
        c = torch.tensor([cap_local], dtype=torch.int64, device=dev)
        dist.all_reduce(c)
        cap_total = int(c.item())
    else:
        cap_total = cap_local
    group = None
    if world > 1:
        group = shard.PeerGroup(rank, world, local_rank, cap_total, n * world)
    else:
        out_m = torch.zeros((cap_total, 3), dtype=torch.int32, device=dev)
        out_o = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    n_jobs = 1 if args.no_overlap else 2
    jobs = [pma.job(local_rank) for _ in range(n_jobs)]
    # the scan stream has priority: when a scan and a placement become runnable together, the persistent scan CTAs
    # (one per SM) are placed first and the placement's small CTAs fill the SMs' remaining thread slots
    st_scan = torch.cuda.Stream(dev, priority=-1)
    st_place = st_scan if args.no_overlap else torch.cuda.Stream(dev, priority=0)
    setup_s = time.time() - t_setup
    kernel_ms, push_ms, timeline = [], [], []

    def finish_prev(s):
        """everything of step s is in its final place (rank 0: from every rank); returns the step's match count"""
        if group is not None:
            tot = group.finish(stream=st_place)
        else:
            tot = jobs[s % n_jobs].wait()
        kernel_ms.append(jobs[s % n_jobs].scan_kernel_ms())
        push_ms.append(jobs[s % n_jobs].push_ms())
        timeline.append(jobs[s % n_jobs].times())
        return tot

    def run(steps, first):
        """steps pipelined steps starting with batch index `first`; returns the last step's total"""
        def scan(s):
            t, o = batches[(first + s) % len(batches)]
            jobs[s % n_jobs].scan(dmode, t, o, cap_local, stream=st_scan)

        def place(s):
            j = jobs[s % n_jobs]
            if group is not None:
                group.place(j, rank * n, rank == world - 1, stream=st_place)
            else:
                j.place(out_m, out_o, stream=st_place)

        return run_pipeline(steps, n_jobs, scan, place, finish_prev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    run(args.warmup, 0)
    barrier()
    n_before = len(sampler.rows)
    kernel_ms.clear()
    push_ms.clear()
    timeline.clear()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches1 = pma.stats()["launches"]
    barrier()
    ev0.record(torch.cuda.current_stream(dev))
    st_scan.wait_stream(torch.cuda.current_stream(dev))
    st_place.wait_stream(torch.cuda.current_stream(dev))
    last_total = run(args.steps, args.warmup)
    torch.cuda.current_stream(dev).wait_stream(st_scan)
    torch.cuda.current_stream(dev).wait_stream(st_place)
    ev1.record(torch.cuda.current_stream(dev))
    barrier()
    time.sleep(0.25)  # let nvidia-smi flush its last samples
    clocks = sampler.stop(skip=n_before)
    clocks["note"] = "nvidia-smi -lms 50 started before the warm-up; the %d samples taken before the timed region are dropped" % n_before
    launches2 = pma.stats()["launches"]
    ms = ev0.elapsed_time(ev1) / args.steps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    my_push = float(np.mean(push_ms)) if push_ms else 0.0
    if world > 1:
        t = torch.tensor([my_push], dtype=torch.float64, device=dev)
        allp_ms = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allp_ms, t)
        push_by_rank = [float(x.item()) for x in allp_ms]
        tl = torch.tensor(timeline[-4:], dtype=torch.float64, device=dev).reshape(-1)
        alltl = [torch.zeros_like(tl) for _ in range(world)]
        dist.all_gather(alltl, tl)
        # per rank, last four steps: ms of (scan start, scan end, push start, push end) relative to the rank's first
        # timed scan start of those four (clocks of different GPUs are not comparable: per-rank offsets only)
        timeline_by_rank = []
        for x in alltl:
            a = x.reshape(-1, 4).cpu().numpy()
            timeline_by_rank.append([[round(float(v - a[0, 0]), 2) if v else None for v in row] for row in a])
    else:
        push_by_rank = []
        timeline_by_rank = []
    job_bytes = step_bytes * world
    value = job_bytes / (ms * 1e-3) / 1e9
    last_batch = (args.warmup + args.steps - 1) % len(batches)
    if args.dump_outputs and rank == 0:
        gm, go = group.result(last_total) if group is not None else (out_m[:last_total], out_o)
        dump_outputs(args.dump_outputs, gm, go, hay_len)

    # ---- in-run parity: the result of the last timed step against the oracle -------------------------------
    # every rank scans a sample of its own shard with the oracle (counts + order-sensitive hashes per haystack,
    # the first quarter of the sample tuple for tuple); the sample is looked up in RANK 0's gathered buffer
    parity = None
    if not args.no_cpu:
        import oracle_api as O

        budget = O.cpu_budget()
        threads = max(1, budget["threads"] // world)
        frac = args.parity_frac if world == 1 else min(args.parity_frac, 0.01)
        ns = max(1, min(n, int(n * frac) if hay_len <= 65536 else max(8, int(n * frac))))
        opma = W.oracle()
        lo = ranges[last_batch][0]
        ptext, poffs = W.host_batch(lo, lo + ns)
        ref = opma.scan_batch(omode, ptext, poffs, nthreads=threads, want_hashes=True)
        nt = max(1, ns // 4)
        ref_t = opma.scan_batch(omode, ptext[: int(poffs[nt])], poffs[: nt + 1], nthreads=threads, want_matches=True)
        mine = {"counts": ref["counts"].astype(np.int64), "hashes": ref["hashes"], "tuples": ref_t["matches"].tobytes(), "nt": nt, "ns": ns}
        if world > 1:
            allp = [None] * world if rank == 0 else None
            dist.gather_object(mine, allp, dst=0)
        else:
            allp = [mine]
        if rank == 0:
            if group is not None:
                gm, go = group.result(last_total)
            else:
                gm, go = out_m[:last_total], out_o
            ok_counts = ok_hash = ok_tuples = True
            checked = 0
            for r, pr in enumerate(allp):
                o = go[r * n: r * n + pr["ns"] + 1].cpu().numpy().astype(np.int64)
                m = gm[int(o[0]): int(o[-1])].cpu().numpy()
                ok_counts &= bool(np.array_equal(np.diff(o), pr["counts"]))
                ok_hash &= bool(np.array_equal(O.hash_matches(m, (o - o[0]).astype(np.uint64)), pr["hashes"]))
                k = int(o[pr["nt"]] - o[0])
                ok_tuples &= m[:k].astype(np.uint32).tobytes() == pr["tuples"]
                checked += pr["ns"]
            total_ok = True
            if world == 1:
                total_ok = last_total == counts[last_batch]
            parity = {"haystacks_checked": checked, "share_of_batch": checked / (n * world), "counts_equal": ok_counts,
                      "hashes_equal": ok_hash, "tuples_equal_first_quarter": ok_tuples, "total_equals_sizing_pass": total_ok,
                      "what": "last timed step, rank 0's %s buffer vs the oracle on every rank's own text" % ("gathered" if world > 1 else "result")}

    # ---- e2e through the host-buffer C-ABI call (pinned host memory), rank-local ------------------------------
    e2e = None
    if not args.no_e2e:
        t0_, o0_ = batches[0]
        ne = n
        try:
            h_text = torch.empty(ne * hay_len, dtype=torch.uint8).pin_memory()
        except RuntimeError:  # the box cannot pin that much: a quarter of the batch
            ne = max(1, n // 4)
            h_text = torch.empty(ne * hay_len, dtype=torch.uint8).pin_memory()
        h_text.copy_(t0_[: ne * hay_len])
        h_offs = (np.arange(ne + 1, dtype=np.uint64) * np.uint64(hay_len))
        h_text_np = h_text.numpy()
        cap = int(counts[0] * (ne / n) * 1.05) + 4096
        # caller-owned result buffers in pinned host memory, reused by every step
        h_out_t = torch.empty(cap * 3, dtype=torch.int32).pin_memory()
        h_out = h_out_t.numpy().view(D.MATCH_DTYPE)
        h_oo_t = torch.empty(ne + 1, dtype=torch.int64).pin_memory()
        h_oo = h_oo_t.numpy().view(np.uint64)
        e2e_ms = []
        if world > 1:
            dist.barrier()
        for i in range(1 + args.e2e_steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = pma.scan_batch_host(dmode, h_text_np, h_offs, out=h_out, out_offs=h_oo)
            dt = time.perf_counter() - t0
            if i >= 1:
                e2e_ms.append(dt * 1e3)
        st = pma.stats()
        e2e_val = ne * hay_len / (np.mean(e2e_ms) * 1e-3) / 1e9
        e2e_ok = int(len(r.matches)) == counts[0] if ne == n else None
        if world > 1:
            t = torch.tensor([e2e_val], dtype=torch.float64, device=dev)
            dist.all_reduce(t)  # sum of per-rank host-buffer throughputs (ranks run concurrently)
            e2e_val = float(t.item())
        e2e = {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(st["h2d_bytes"]),
               "d2h_bytes_per_step": int(st["d2h_bytes"]), "ms_per_step": float(np.mean(e2e_ms)),
               "matches_per_step": int(len(r.matches)), "match_count_equals_device_path": e2e_ok,
               "workload": "%d of the step batch's %d haystacks x %d B per GPU through dach_scan_batch_host: pinned host text -> "
                           "device -> scan -> pinned host matches, 64 MiB slices, uploads two slices ahead" % (ne, n, hay_len)}
        del h_text, h_out_t, h_oo_t

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the scan kernel) ------------------------------------------------
    peak, peak_src = measured_peaks()
    k_ms = float(np.mean(kernel_ms))
    achieved = step_bytes / (k_ms * 1e-3) / 1e9
    kname = {"C3": "k_scan_machine<StdMachine3<M_OVERLAPPING>, Lane3, 1024, 1, false>", "C3-find": "k_scan_machine<StdMachine3<M_FIND>, Lane3, 1024, 1, false>",
             "C2": "k_scan_machine<StdMachine3<M_OVERLAPPING>, Lane3, 1024, 1, false>", "C5": "k_scan_machine<StdMachine3<M_OVERLAPPING>, Lane3, 1024, 1, false>",
             "C4": "k_scan_machine<CwMachine<M_LEFTMOST>, LaneCw, 1024, 1, false>",
             "C4-bw": "k_scan_machine<LmMachine, LaneLm, 1024, 1, false>"}[args.config]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": kname, "kernel_ms": k_ms,
                "algorithmic_bytes_per_launch": step_bytes, "peak_source": peak_src,
                "note": "algorithmic bytes = 1 B read per haystack byte x bytes per launch (DESIGN.md); kernel_ms = mean CUDA-event "
                        "time of the scan kernel over the timed steps (events on its launch stream, inside the library)"}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            ent = tj.get(args.config) or (tj if args.config == "C3" and "dram_bytes_per_byte_scanned" in tj else None)
            if ent and ent.get("dram_bytes_per_byte_scanned") is not None:
                roofline["traffic"] = ent["dram_bytes_per_byte_scanned"] * step_bytes
                roofline["traffic_source"] = ent.get("source", "profiles/traffic.json (ncu --set full capture of this kernel)")
        except Exception:
            pass

    # ---- CPU baseline: the C port on the host cores, bounded sample -------------------------------------------
    cpu = None
    if not args.no_cpu and world == 1:  # the CPU baseline is reported on rank 0 at N = 1 only
        import oracle_api as O

        budget = O.cpu_budget()
        threads = budget["threads"]
        nc = min(n, max(threads * 4, (1 << 30) // hay_len))  # about 1 GiB of the batch
        v_all, dt, reps, _, nbytes = cpu_sample(W, opma, omode, nc, 10.0, threads)
        v_one, _, _, _, _ = cpu_sample(W, opma, omode, max(64 if hay_len <= 8192 else 4, nc // max(threads, 1)), 2.0, 1)
        cpu = {"value": v_all, "unit": UNIT, "cores": threads, "kind": "port", "single_thread": v_one, "cpu": budget,
               "sample": "first %d haystacks x %d B (%.0f MiB) of rank 0's batch, %d passes, %d pinned threads, %.2f s per pass" % (
                   nc, hay_len, nbytes / 2**20, reps, threads, dt),
               "note": "C restatement of daachorse 4.0.0's scan loops on the crate's array-of-structs records, -O3 -march=native "
                       "built on this box, persistent pinned threads, matches stored to a per-thread ring (Rust toolchain "
                       "unavailable: the crate itself cannot be built here)"}
    if cpu is not None:
        cpu["parity"] = parity
    elif parity is not None:
        cpu = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": "N > 1: parity only", "parity": parity}

    line = {
        "metric": metric_name(W.spec), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": "%s: %s, %s, %d haystacks x %d B per GPU per step (seeded windows of a %d MiB text pool, "
                               "materialised in HBM; %d batch(es) resident, %.2f GiB per GPU)" % (
                                   args.config, W.spec["what"], W.mode_name, n, hay_len, len(W.pool) >> 20, len(batches), resident / 2**30),
                   "n_patterns": len(W.ps), "num_states": pma.num_states(), "automaton_heap_mib": pma.heap_bytes() / 2**20,
                   "image_mib": pma.stats()["image_bytes"] / 2**20, "hay_len": hay_len, "haystacks_per_gpu": n,
                   "bytes_per_gpu": step_bytes, "matches_per_step_per_gpu": counts[last_batch],
                   "matches_per_byte": counts[last_batch] / step_bytes,
                   "l2": "inputs of consecutive steps (%.2f GiB per GPU before one repeats) are larger than L2 (126 MB); no flush needed" % (
                       resident / 2**30),
                   "parallelism": "haystack shards, one rank per GPU" + (
                       "; every rank's placement kernel stores its matches into rank 0's dense buffer over NVLink peer memory "
                       "(dach_group_*), rank 0 holds the rebased %d-GPU result after every step" % world if world > 1 else ""),
                   "pipelining": "none (--no-overlap)" if args.no_overlap else "two jobs: the placement of step s runs beside the scan of step s+1",
                   "peer_push_ms_by_rank": push_by_rank, "timeline_last4_by_rank": timeline_by_rank,
                   "options": args.option, "setup_s": setup_s},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": int(launches2 - launches1), "launches_per_step": (launches2 - launches1) / args.steps,
        "clocks": clocks,
    }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.stdout.flush()
    if saved_stdout is not None:
        os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
