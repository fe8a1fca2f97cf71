"""`bench.py --dump-outputs DIR`: the windows the last timed step of the device-resident sliding-window path emitted,
written as DIR/<column>.npy so that two builds can be compared output for output on the same seeded inputs."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench as B  # noqa: E402


def _args(*argv):
    saved = sys.argv
    sys.argv = ["bench.py", *argv]
    try:
        return B.parse()
    finally:
        sys.argv = saved


def _written(d):
    """The files of a dump, int64 columns put back together from their two halves."""
    got = {f[:-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    assert all(a.dtype == np.float64 for a in got.values())
    for name in [f[:-len("_hi")] for f in got if f.endswith("_hi")]:
        hi, lo = got.pop(name + "_hi"), got.pop(name + "_lo")
        assert np.all((lo >= 0) & (lo < 2**32) & (hi == np.round(hi)))
        got[name] = (hi.astype(np.int64) << 32) + lo.astype(np.int64)
    return got


def test_dump_writes_every_value_exactly_as_float64(tmp_path):
    rng = np.random.default_rng(0)
    cols = {c: rng.integers(-2**63, 2**63 - 1, 1000, dtype=np.int64, endpoint=True) for c in B.OUT_COLS}
    cols["key"][:4] = [-2**63, -1, 0, 2**63 - 1]
    cols["_timestamp"][:] = 1_700_000_060 * 10**9 - 1  # window end - 1 ns: no float64 holds it
    cols["avg"] = rng.random(1000)
    B.dump_outputs(str(tmp_path), cols)
    assert sorted(os.listdir(tmp_path)) == sorted(["avg.npy"] + [f"{c}_{h}.npy" for c in B.OUT_COLS if c != "avg"
                                                                 for h in ("hi", "lo")])
    got = _written(tmp_path)
    assert set(got) == set(B.OUT_COLS)
    for name, a in got.items():
        assert a.dtype == cols[name].dtype and np.array_equal(a, cols[name])


def test_dump_above_the_limit_keeps_one_seeded_sample_of_rows(tmp_path, monkeypatch):
    monkeypatch.setattr(B, "DUMP_BYTES", 200_000)
    n = 100_000
    cols = {c: np.arange(n, dtype=np.int64) + i * n for i, c in enumerate(B.OUT_COLS)}
    cols["avg"] = np.arange(n, dtype=np.float64) + 4 * n
    for d in ("a", "b"):
        B.dump_outputs(str(tmp_path / d), cols)
    a, b = _written(tmp_path / "a"), _written(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= B.DUMP_BYTES
    rows = a["key"]
    assert 0 < len(rows) < n and np.all(np.diff(rows) > 0)
    for i, c in enumerate(B.OUT_COLS):
        assert np.array_equal(a[c], rows + i * n)  # the same rows of every column
        assert np.array_equal(a[c], b[c])  # and the same rows from run to run


def test_dump_outputs_is_refused_outside_the_sliding_path_of_one_gpu(monkeypatch):
    assert _args("--dump-outputs", "d").dump_outputs == "d"
    for argv in (["--workload", "join"], ["--workload", "session"], ["--impl", "reference"]):
        with pytest.raises(SystemExit):
            _args("--dump-outputs", "d", *argv)
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(SystemExit):
        _args("--dump-outputs", "d")


@pytest.mark.gpu
def test_dumped_columns_are_the_last_window_the_timed_steps_emitted():
    """The host columns device_resident hands back are the last window of the timed steps, checksum for checksum as
    the verify pass reduces that window on the device, one row per key in key order."""
    import torch

    from arroyo_b200 import ffi, operators as native

    args = _args("--rows-per-pane", str(1 << 20), "--keys", str(1 << 16))
    device = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    torch.cuda.set_stream(torch.cuda.Stream(device=device))
    W, K, rows = B.steady_warmup(0), 2, args.rows_per_pane
    gen = B.make_generator(torch, device, rows, args.keys, args.dist, 42, args.keyspace)
    panes = [gen(p) for p in range(W + K)]
    last = {}
    _, _, _, _, sums = B.device_resident(args, torch, native, ffi, 0, panes, W, K, rows, collect=True,
                                         last_window=last)
    ws = max(sums)
    we, n, cnt, sm, av = sums[ws]
    assert set(last) == set(B.OUT_COLS) and len(last["key"]) == n == args.keys
    assert np.all(last["window_start"] == ws) and np.all(last["window_end"] == we)
    assert np.all(last["_timestamp"] == we - 1)
    assert np.all(np.diff(last["key"]) > 0)
    assert int(last["count"].sum()) == cnt == 10 * rows
    assert int(last["sum"].sum()) & ((1 << 64) - 1) == sm
    assert abs(float(last["avg"].sum()) - av) <= 1e-9 * abs(av)
