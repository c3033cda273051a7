"""Host logic of bench.py that needs no GPU: the order in which a pipelined run issues scans, placements and
finishes (a wrong order deadlocks a shard group or reuses a job that is still placing), the batch windows of every
config, the --dump-outputs writer, the CPU budget."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import oracle_api as O  # noqa: E402


@pytest.mark.parametrize("n_jobs", [1, 2])
@pytest.mark.parametrize("steps", [0, 1, 2, 3, 7])
def test_pipeline_order(n_jobs, steps):
    log = []
    busy = {}      # job index -> step it currently holds (scanned, not yet finished)

    def scan(s):
        j = s % n_jobs
        assert j not in busy, "job %d reused for step %d while step %d is not finished" % (j, s, busy.get(j))
        busy[j] = s
        log.append(("scan", s))

    def place(s):
        assert busy.get(s % n_jobs) == s and ("scan", s) in log and ("place", s) not in log
        if n_jobs > 1 and s + 1 < steps:
            assert ("scan", s + 1) in log, "the next scan must be enqueued before place() may block"
        log.append(("place", s))

    def finish(s):
        assert ("place", s) in log and ("finish", s) not in log
        del busy[s % n_jobs]
        log.append(("finish", s))
        return 100 + s

    tot = bench.run_pipeline(steps, n_jobs, scan, place, finish)
    assert tot == (100 + steps - 1 if steps else 0)
    assert not busy
    for kind in ("scan", "place", "finish"):
        assert [s for k, s in log if k == kind] == list(range(steps))


def test_batch_windows_of_every_config():
    class W(bench.Workload):
        def __init__(self, name, n_total, window):  # no pattern / pool generation
            self.spec = bench.CONFIGS[name]
            self.n_total = n_total
            self.window = window

    for name in bench.CONFIGS:
        spec = bench.CONFIGS[name]
        if "window" in spec:
            w = W(name, 12800, 1024)
            r = w.batch_ranges()
            assert len(r) == 13 and r[0] == (0, 1024) and r[11] == (11264, 12288) and r[12] == (11776, 12800)
            assert all(hi - lo == 1024 for lo, hi in r)
            covered = set()
            for lo, hi in r:
                covered.update(range(lo, hi, 512))
            assert covered == set(range(0, 12800, 512))       # the whole 12.5 GiB shard is scanned
            assert W(name, 1280, 1024).batch_ranges() == [(0, 1024), (256, 1280)]   # --scale 0.1
            assert W(name, 512, 512).batch_ranges() == [(0, 512)]
        else:
            w = W(name, 10 * spec["batches"], 10)
            assert w.batch_ranges() == [(10 * k, 10 * k + 10) for k in range(spec["batches"])]


@pytest.mark.parametrize("n,hay_len,most", [(1, 4096, 3), (300, 4096, 3), (70000, 64, 40), (3 << 20, 1 << 20, 2)])
def test_dump_outputs(tmp_path, n, hay_len, most):
    """--dump-outputs: float64 arrays, the sampled haystacks' matches exactly as the result holds them, the same
    files for the same result, and the size bound however many haystacks and matches there are."""
    import numpy as np
    import torch

    rng = np.random.default_rng(n)
    counts = rng.integers(0, most + 1, size=n)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    m = torch.from_numpy(rng.integers(-2**31, 2**31, size=(int(offs[-1]), 3), dtype=np.int64).astype(np.int32))
    o = torch.from_numpy(offs)
    bench.dump_outputs(str(tmp_path / "a"), m, o, hay_len)
    bench.dump_outputs(str(tmp_path / "b"), m, o, hay_len)
    names = ["match_counts.npy", "match_haystacks.npy", "matches.npy", "offsets.npy"]
    assert sorted(os.listdir(tmp_path / "a")) == names
    got = {nm[:-4]: np.load(tmp_path / "a" / nm) for nm in names}
    assert all(a.dtype == np.float64 for a in got.values())
    assert all(np.array_equal(a, np.load(tmp_path / "b" / nm)) for nm, a in zip(names, got.values()))
    assert sum(os.path.getsize(tmp_path / "a" / nm) for nm in names) <= 64 << 20
    stride = -(-(n + 1) // bench.DUMP_OFFSETS_MAX)
    assert np.array_equal(got["offsets"], offs[::stride])
    hs = got["match_haystacks"].astype(np.int64)
    assert len(hs) == min(n, bench.DUMP_HAYSTACKS_MAX, bench.DUMP_TEXT_BYTES // hay_len)
    assert np.all(np.diff(hs) > 0) and np.array_equal(got["match_counts"], counts[hs])
    want = np.concatenate([m.numpy()[offs[h]: offs[h + 1]] for h in hs]).view(np.uint32)[: bench.DUMP_MATCHES_MAX]
    assert np.array_equal(got["matches"], want)


def test_cpu_budget_is_sane():
    b = O.cpu_budget()
    assert 1 <= b["threads"] <= b["affinity"] <= max(b["os_cpu_count"], b["affinity"])
    assert b["cgroup_cpu_quota"] is None or b["cgroup_cpu_quota"] > 0


def test_metric_names_follow_baseline_json():
    import json

    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert bench.metric_name(bench.CONFIGS["C3"]) in base["metric"] or "find_overlapping_iter, 675k-pat bytewise" in base["metric"]
    assert bench.metric_name(bench.CONFIGS["C3"]) == "input GB/s scanned, find_overlapping_iter, 675k-pat bytewise"
