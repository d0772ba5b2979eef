"""bench.py helpers that need no GPU: the nvidia-smi sampler (started before the warm-up, armed at the first timed
step) against a stub `nvidia-smi`, the CPU arm's bookkeeping, and the --dump-outputs writer."""
import importlib.util
import os
import stat
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


STUB = """#!/bin/bash
i=0
while true; do
  echo "0, $((1900 + i)), 1965, 300.5, 0x0000000000000000, Not Active, Not Active, Not Active, %s"
  i=$((i+1)); sleep 0.05
done
"""


def _install_stub(tmp_path, monkeypatch, power_cap="Not Active"):
    exe = tmp_path / "nvidia-smi"
    exe.write_text(STUB % power_cap)
    exe.chmod(exe.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ["PATH"])


def test_clock_sampler_counts_from_the_armed_point(tmp_path, monkeypatch):
    _install_stub(tmp_path, monkeypatch)
    b = _bench()
    s = b.ClockSampler(0)
    s.start()
    time.sleep(0.45)                    # "warm-up": these samples are not reported
    s.arm()
    time.sleep(0.3)
    out = s.stop()
    assert 4 <= out["samples"] <= 9, out            # 0.3 s at 50 ms + the one just before arm()
    assert out["sm_mhz"] >= 1905 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == []


def test_clock_sampler_reports_power_cap_and_survives_a_missing_tool(tmp_path, monkeypatch):
    _install_stub(tmp_path, monkeypatch, power_cap="Active")
    b = _bench()
    s = b.ClockSampler(0)
    s.arm()                             # arm() alone starts the process
    time.sleep(0.25)
    assert s.stop()["reasons"] == ["sw_power_cap"]
    monkeypatch.setenv("PATH", str(tmp_path / "nowhere"))
    s2 = b.ClockSampler(0)
    s2.start()
    s2.arm()
    assert s2.stop()["reasons"] == ["nvidia-smi unavailable"]


def _match_list(n, seed):
    rng = np.random.default_rng(seed)
    cnt = rng.integers(1, 30, size=n)
    r = np.repeat(np.arange(n), cnt)
    k = np.arange(len(r)) - np.repeat(np.cumsum(cnt) - cnt, cnt)           # position inside the row
    c = (r * 7919 + 37 * k) % n                                             # (row, col) pairs are unique
    s = rng.random(len(r))
    o = rng.permutation(len(r))                      # the dump sorts by (row, col) itself
    return r[o], c[o], s[o]


def test_dump_outputs_writes_every_pair_of_a_seeded_row_sample(tmp_path, monkeypatch):
    b = _bench()
    n = 5000
    r, c, s = _match_list(n, 1)
    monkeypatch.setattr(b, "DUMP_SAMPLE_ROWS", 1000)
    b.dump_outputs(str(tmp_path / "a"), (r, c, s), n)
    b.dump_outputs(str(tmp_path / "b"), (r[::-1], c[::-1], s[::-1]), n)
    got = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(got) == ["col.npy", "pairs_per_row.npy", "row.npy", "sample_rows.npy", "score.npy"]
    for f, a in got.items():
        assert a.dtype == np.float64, f
        assert np.array_equal(a, np.load(tmp_path / "b" / f)), f          # same pairs in any order: same files
    assert np.array_equal(got["pairs_per_row.npy"], np.bincount(r, minlength=n))
    rows = got["sample_rows.npy"].astype(np.int64)
    assert len(rows) == 1000 and np.all(np.diff(rows) > 0)
    keep = np.isin(r, rows)
    want = sorted(zip(r[keep].tolist(), c[keep].tolist(), s[keep].tolist()))
    have = list(zip(got["row.npy"].astype(np.int64).tolist(), got["col.npy"].astype(np.int64).tolist(),
                    got["score.npy"].tolist()))
    assert have == want


def test_dump_outputs_stays_within_the_byte_budget(tmp_path, monkeypatch):
    b = _bench()
    n = 5000
    r, c, s = _match_list(n, 2)
    monkeypatch.setattr(b, "DUMP_BYTES", 400_000)
    b.dump_outputs(str(tmp_path), (r, c, s), n)
    total = sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path))
    assert 300_000 < total <= 400_000, total
    rows = np.load(tmp_path / "sample_rows.npy").astype(np.int64)
    full = np.random.default_rng(0).permutation(n)[:len(rows)]            # a prefix of the seeded permutation
    assert np.array_equal(rows, np.sort(full))
    assert len(np.load(tmp_path / "row.npy")) == np.isin(r, rows).sum()
