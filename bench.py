#!/usr/bin/env python
"""bench.py -- rows/sec of the sliding-window SUM/AVG hot path (BASELINE.json config 3) on N B200s.

Workload (`config.workload`): hop(1 s slide, 10 s width) SUM(value), AVG(value), COUNT(*) GROUP BY key,
1 048 576 distinct i64 keys (uniform), Arrow-shaped batches of 65 536 rows [key i64, value i64,
_timestamp ts-ns], 16 Mi rows per 1-s pane (256 batches), Nexmark bounded disorder (groups of 50),
watermark = batch-min timestamp - 1 s at most once per second of event time (SURVEY.md 8(d)).

A *step* = one pane: 256 batches through process_batch + the watermark that closes one pane and emits
one 10-s window (<= 1 Mi rows x 6 columns).

  value     device-resident: inputs already in HBM, windows left in HBM (process_device_batches /
            handle_watermark_device of the C ABI); timed with CUDA events on the operator's stream
  e2e       the same through the reference-facing call with HOST buffers: pinned Arrow batches in via
            arroyo_b200_op_process_batch, emitted windows out as host Arrow batches
  roofline  the ingest (window-assign + partial aggregate: part_kernel + agg_kernel per launch): 24 algorithmic
            bytes per input row / the CUDA-event time of the step's ingest launches, against the measured HBM
            copy bandwidth (MEASURED_PEAKS.json); `traffic` = DRAM bytes from the committed ncu capture
  verified  the windows of a second, identical pass over the panes the CPU baseline consumed equal the C
            oracle's, checksum by checksum (rows out, sum COUNT, wrapping sum SUM bit-exact; sum AVG 1e-6);
            a mismatch makes the script exit non-zero
  cpu_baseline / --impl reference
            the C restatement of the reference's algorithm (oracle/window_oracle.c, "port": the Rust
            reference cannot be built here) on all host cores, key-partitioned like the reference

Multi-GPU (N > 1): one process per GPU; every rank ingests its own shard of the stream (seed 42 + rank),
pre-aggregates it per pane, hash-partitions the partial rows on the device, exchanges them over NCCL (the
library's own round: csrc/exchange.cu) and the owner of a key merges and emits (weak scaling: per-GPU
input fixed; arroyo_b200/multi_gpu.py).  `--workload join | session`: BASELINE configs[3] / configs[4]
(bench_workloads.py).
"""
import os as _os

if int(_os.environ.get("WORLD_SIZE", "1")) > 4:
    # Two NCCL communicators live in every rank at N > 1 (torch.distributed's and the Shuffle edge's own,
    # csrc/exchange.cu); all this job moves through collectives is an 80-byte control record per round, so NVLink SHARP
    # (NVLS: multicast objects set up per communicator across the whole NVSwitch domain) buys nothing and is left out
    # of the set-up on large boxes.  The one N = 8 attempt of round 2 printed nothing within five minutes (cause not
    # established: no GPU time was left to look; DESIGN.md section 7); N <= 4 run with NCCL's defaults, as measured.
    _os.environ.setdefault("NCCL_NVLS_ENABLE", "0")

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

S = 1_000_000_000
T0 = 1_700_000_000 * S
BATCH_ROWS = 65_536
WIDTH, SLIDE, WM_DELAY = 10 * S, 1 * S, 1 * S
KEY_MULT = 0x9E3779B97F4A7C15  # odd => bijection on u64: keys are scattered over the i64 range


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--keys", type=int, default=1 << 20)
    ap.add_argument("--rows-per-pane", type=int, default=1 << 24)
    ap.add_argument("--dist", default="uniform", choices=["uniform", "hot"])
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--remerge", action="store_true", help="re-merge all panes per slide (reference algorithm)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--no-combine", action="store_true", help="measurement knob: no warp-combining of equal keys")
    ap.add_argument("--avg-f64", action="store_true", help="measurement knob: AVG with its own f64 accumulator")
    ap.add_argument("--chunk-log2", type=int, default=0, help="rows per ingest launch = 2^n (default 24)")
    ap.add_argument("--keyspace", default="scattered", choices=["scattered", "dense"],
                    help="scattered: key ids multiplied by an odd 64-bit constant (every key is hashed); "
                         "dense: Nexmark-shaped ids 1000 + n (the operator maps the range straight onto dense ids)")
    ap.add_argument("--e2e-host", default="library", choices=["library", "python"],
                    help="e2e run loop: arroyo_b200_op_run_batches (the loop a compiled shim would run, inside the "
                         "library) or one ctypes call per batch from Python")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="do not bind the process to the CPUs local to its GPU (NVML affinity)")
    ap.add_argument("--e2e-trials", type=int, default=3, help="e2e passes (median reported, all listed)")
    ap.add_argument("--skip-pageable", action="store_true", help="e2e: skip the extra pass over pageable host buffers")
    ap.add_argument("--sync-emit", action="store_true",
                    help="e2e: blocking arroyo_b200_op_handle_watermark instead of the begin / poll pair")
    ap.add_argument("--no-direct", action="store_true", help="accepted and ignored (every key is hashed since round 2)")
    ap.add_argument("--one-pass", action="store_true",
                    help="measurement knob: the one-pass ingest kernel (probe + REDs per row) instead of the two-pass ingest")
    ap.add_argument("--local-chunk-log2", type=int, default=24,
                    help="N>1, partials: rows per ingest launch of the local stage = 2^n (one pane per launch: the two-pass "
                         "ingest pays its per-launch table builds once; 2^23 measured 0.73 vs 0.53 ms per step, "
                         "profiles/r02_partials_n1_c2*.json)")
    ap.add_argument("--python-exchange", action="store_true",
                    help="N>1, partials: the shuffle round through torch.distributed (device partitioner + all_gather + "
                         "all_to_all_single from Python) instead of the library's own round (csrc/exchange.cu: partition + "
                         "control all-gather + grouped ncclSend / ncclRecv in one C call): 56.7 vs 61.9 G rows/s at N = 2 "
                         "(profiles/r02_bench_n2*.json)")
    ap.add_argument("--native-exchange", action="store_true",
                    help="N>1, partials: the library's own round (see --python-exchange).  It is the default up to 4 GPUs, "
                         "where it was measured; above that the default is the torch.distributed round, the one that has "
                         "run on eight GPUs (round 1) -- the library's round is selected with this flag")
    ap.add_argument("--sync-plan", action="store_true",
                    help="N>1, partials: run the local stage, the shuffle and the owner stage in sequence on one host "
                         "thread instead of as a two-stage pipeline")
    ap.add_argument("--workload", default="sliding", choices=["sliding", "join", "session"],
                    help="sliding = the headline (BASELINE configs[2]); join = configs[3] (q8-shaped windowed hash join "
                         "behind two key-hash shuffles); session = configs[4] (session windows behind a key-hash shuffle): "
                         "bench_workloads.py")
    ap.add_argument("--join-persons-log2", type=int, default=21, help="--workload join: persons per GPU and window = 2^n")
    ap.add_argument("--join-auctions-log2", type=int, default=23, help="--workload join: auctions per GPU and window = 2^n")
    ap.add_argument("--session-keys", type=int, default=10_000_000, help="--workload session: keys per GPU")
    ap.add_argument("--session-rows-log2", type=int, default=22, help="--workload session: rows per GPU and step = 2^n")
    ap.add_argument("--session-split", type=int, default=1,
                    help="--workload session, N = 1, measurement knob: hand every step over as this many batches that cover "
                         "the same second, i.e. what an owner behind that many senders receives")
    ap.add_argument("--shuffle", default="partials", choices=["partials", "rows"],
                    help="N>1: what crosses the all-to-all (per-pane partial aggregates, or raw rows)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the windows the last timed step emitted under DIR as float64 "
                         ".npy files, exactly (avg.npy; <column>_hi.npy / <column>_lo.npy = upper / lower 32 bits of "
                         "every int64 column), rows ordered by window and key, a seeded row sample above 64 MB: the "
                         "sliding workload at N = 1")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.workload != "sliding" or args.impl != "ours" or world > 1):
        ap.error("--dump-outputs writes the device-resident sliding-window path of one GPU: "
                 "--workload sliding --impl ours at N = 1")
    args.native_exchange = (not args.python_exchange) and (world <= 4 or args.native_exchange)
    return args


# ------------------------------------------------------------------------------------------------
# synthetic Nexmark-bid-shaped input (generated on the device; seed 42 + rank)
# ------------------------------------------------------------------------------------------------
POOL = 8  # distinct (key, value) panes; every step still gets its own timestamps


def make_generator(torch, device, rows_per_pane, n_keys, dist, seed, keyspace="scattered"):
    """pane(p) -> (key, value, ts) device tensors of the p-th 1-s pane.  Keys / values cycle through a pool of
    POOL independently drawn panes (the operator never sees the same timestamps twice)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    i = torch.arange(rows_per_pane, device=device, dtype=torch.int64)
    # event i of a pane happens at i * (1 s / rows_per_pane); events are permuted inside groups of 50
    # (nexmark/operator.rs:515-521 out_of_order_group_size)
    grp = (i // 50).to(torch.float64) + torch.rand(rows_per_pane, device=device, generator=g, dtype=torch.float64) * 0.999
    order = torch.argsort(grp)
    offs = (order * S) // rows_per_pane
    del grp, order, i
    pool = []
    for j in range(POOL):
        kid = torch.randint(0, n_keys, (rows_per_pane,), device=device, generator=g, dtype=torch.int64)
        if dist == "hot":  # 75 % of the rows on the current hot id (nexmark hot_bidders_ratio 4 -> 3 of 4 rows)
            hot = torch.rand(rows_per_pane, device=device, generator=g) < 0.75
            kid = torch.where(hot, torch.full_like(kid, (j // 4) % n_keys), kid)
        if keyspace == "dense":
            key = kid + 1000  # nexmark FIRST_PERSON_ID / FIRST_AUCTION_ID style surrogate ids
        else:
            key = kid * torch.tensor(KEY_MULT - (1 << 64), dtype=torch.int64, device=device)  # wrapping multiply
        # price = floor(10^U(0,6) * 100)  (nexmark/operator.rs:643-645)
        u = torch.rand(rows_per_pane, device=device, generator=g, dtype=torch.float64) * 6.0
        val = torch.floor(torch.pow(10.0, u) * 100.0).to(torch.int64)
        pool.append((key, val))
        del kid, u

    def pane(p):
        key, val = pool[p % POOL]
        return key, val, offs + (T0 + p * SLIDE)

    return pane


def watermark_schedule(ts_min_max):
    """Simulates the WatermarkGenerator over the per-batch (min, max) timestamps: returns, per batch,
    the watermark it broadcasts after the batch (or None)."""
    from arroyo_b200 import WatermarkGenerator
    gen = WatermarkGenerator(WM_DELAY)
    return [gen.on_batch(mn, mx) for mn, mx in ts_min_max]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region.  The sampler process is started before
    the warm-up (nvidia-smi needs tens of milliseconds to print its first line, longer than a 20-step timed region);
    every line is stamped on arrival and `stop()` keeps the ones that arrived inside [begin(), end()]."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 5

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []  # (arrival time, text)
        self.t0 = self.t1 = None

    def start(self, wait_first_s=3.0):
        """Starts the sampler and waits (bounded) for its first line: nvidia-smi needs ~0.1 s to print it -- longer than
        the warm-up plus a 100-step timed region -- and from then on prints one every PERIOD_MS.  It is started right
        before the warm-up, not earlier: polling through the job's set-up (allocations, NCCL initialisation) contends
        with those calls for the driver."""
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", str(self.PERIOD_MS)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            deadline = time.perf_counter() + wait_first_s
            while not self.lines and time.perf_counter() < deadline and self.proc.poll() is None:
                time.sleep(0.005)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        if self.t1 is None:
            self.end()
        time.sleep(2.5 * self.PERIOD_MS * 1e-3)  # the sample that was being taken when the region ended
        deadline = time.perf_counter() + 1.0
        while not self.lines and time.perf_counter() < deadline:  # nvidia-smi still starting up: its first sample then
            time.sleep(0.01)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0 = self.t0 if self.t0 is not None else 0.0
        slack = 2.0 * self.PERIOD_MS * 1e-3  # a line describes the period that ended when it was printed
        inside = [ln for (t, ln) in self.lines if t0 <= t <= self.t1 + slack]
        note = None
        if not inside and self.lines:
            # region shorter than the sampling period: the sample nearest to it
            inside = [min(self.lines, key=lambda x: abs(x[0] - self.t1))[1]]
            note = "timed region shorter than the sampling period: nearest sample"
        sm, mx, reasons = [], None, set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
               "samples": len(sm)}
        if note:
            out["note"] = note
        return out


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def ncu_traffic():
    """dram bytes per ingest launch from the committed ncu capture (profiles/), or None."""
    p = os.path.join(ROOT, "profiles", "ingest_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def op_flags(args):
    from arroyo_b200 import ffi
    return ((ffi.FLAG_REMERGE_ONLY if args.remerge else 0) | (ffi.FLAG_NO_COMBINE if args.no_combine else 0) |
            (ffi.FLAG_AVG_F64 if args.avg_f64 else 0) | (ffi.FLAG_NO_TWO_PASS if args.one_pass else 0))


def steady_warmup(requested, extra=0):
    """Warm-up panes actually run: never fewer than one full window (width / slide panes) plus the pipeline lag and a
    margin, whatever --warmup says.  The timed region must see the steady state (every pane of the window resident,
    the running window primed, all buffers allocated); with fewer warm-up panes it times the cold start instead."""
    return max(int(requested), WIDTH // SLIDE + 3 + extra)


def workload_config(args, world):
    """`config` of the JSON line: identical for both arms (--impl ours / reference)."""
    rows = args.rows_per_pane
    return {"workload": "BASELINE configs[2]: hop(1s slide,10s width) SUM/AVG/COUNT GROUP BY key, "
                        f"{args.keys} i64 keys ({args.dist}, {args.keyspace}); every GPU's source shard delivers {rows} "
                        f"rows per 1-s pane in {rows // BATCH_ROWS} Arrow-shaped batches of {BATCH_ROWS}; 1 step = 1 pane "
                        "ingested per GPU + the 10-s window it closes emitted",
            "keys": args.keys, "rows_per_step_per_gpu": rows, "batch_rows": BATCH_ROWS, "width_s": WIDTH // S,
            "slide_s": SLIDE // S, "dist": args.dist, "keyspace": args.keyspace, "n_gpus": world,
            "parallelism": "1 gpu" if world == 1 else f"key-partitioned x{world} (key-hash shuffle, NCCL all-to-all)",
            "l2": f"inputs larger than L2 ({rows * 24 // 1000000} MB per step per GPU, never re-read)"}


def window_config():
    import arroyo_b200 as ab
    return ab.WindowAggConfig(width=WIDTH, slide=SLIDE, key_names=["key"],
                              aggs=[ab.Agg("sum", "value", "sum"), ab.Agg("avg", "value", "avg"),
                                    ab.Agg("count", None, "count")], window_index=1)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the C restatement on the host cores
# ------------------------------------------------------------------------------------------------
def host_panes(torch, gen_pane, n):
    out = []
    for p in range(n):
        k, v, t = gen_pane(p)
        out.append((k.cpu().numpy(), v.cpu().numpy(), t.cpu().numpy()))
    return out


def sample_pane(torch, device, pane, n_rows):
    """The bounded sample of one pane: whole BATCH_ROWS-row batches dropped uniformly (every batch keeps its shape).
    n_rows == the pane's row count returns the pane itself."""
    k, v, t = pane
    rows = k.numel()
    if n_rows >= rows:
        return k, v, t
    nb = rows // BATCH_ROWS
    keep = torch.linspace(0, nb - 1, n_rows // BATCH_ROWS, device=device).round().to(torch.int64)
    idx = (keep[:, None] * BATCH_ROWS + torch.arange(BATCH_ROWS, device=device)[None, :]).reshape(-1)
    return k[idx], v[idx], t[idx]


def run_cpu(torch, args, device, budget_s, warm_panes, timed_panes, seeds=(42,)):
    """Times the oracle port on all host cores over `timed_panes` panes after `warm_panes` warm-up panes.
    If a full pane is too slow for the budget the panes carry fewer rows (bounded sample).  `seeds`: the source
    shards whose union the subtasks consume (one per GPU of the run being checked).  Also returns the per-window
    checksums of everything it emitted: the GPU verify pass runs the same panes and must reproduce them."""
    from oracle import c_oracle
    threads = c_oracle.load().oracle_max_threads()
    threads = max(1, min(threads, 1024))
    rows = args.rows_per_pane
    r = c_oracle.Runner(threads, WIDTH, SLIDE, WM_DELAY, BATCH_ROWS)
    total = warm_panes + timed_panes
    step_s = []
    n_rows = rows
    gens = {}

    def pane_of(seed, p):
        # one generator (2 GB of pooled keys / values) alive at a time
        if seed not in gens:
            gens.clear()
            torch.cuda.empty_cache() if device.type == "cuda" else None
            gens[seed] = make_generator(torch, device, rows, args.keys, args.dist, seed, args.keyspace)
        return gens[seed](p)

    # pane 0 at full size calibrates the sample
    dt0 = 0.0
    for seed in seeds:
        k, v, t = [x.cpu().numpy() for x in pane_of(seed, 0)]
        dt0 += r.feed(k, v, t)
    est = dt0 * 2.5  # later panes also pay a 10-pane merge per slide
    if est * (total - 1) > budget_s:
        frac = max(budget_s / (est * (total - 1)), 1.0 / 64)
        n_rows = max(BATCH_ROWS, int(rows * frac) // BATCH_ROWS * BATCH_ROWS)
    if n_rows < rows:
        # the calibration pane does not belong to the sampled stream: start over
        r.close()
        r = c_oracle.Runner(threads, WIDTH, SLIDE, WM_DELAY, BATCH_ROWS)
        first = 0
    else:
        first = 1
    for p in range(first, total):
        dt = 0.0
        for seed in seeds:
            k, v, t = sample_pane(torch, device, pane_of(seed, p), n_rows)
            dt += r.feed(k.cpu().numpy(), v.cpu().numpy(), t.cpu().numpy())
        if p >= warm_panes:
            step_s.append(dt)
    res = r.result()
    windows = r.windows()
    r.close()
    gens.clear()
    secs = sum(step_s)
    return {"rows_per_s": len(seeds) * n_rows * len(step_s) / secs, "threads": threads, "rows_per_step": n_rows,
            "steps": len(step_s), "ms_per_step": 1e3 * secs / len(step_s), "rows_out": int(res.rows_out),
            "windows": windows, "panes": total, "seeds": list(seeds),
            "sample": (f"{len(step_s)} panes x {len(seeds)} shard(s) x {n_rows} rows ({n_rows // BATCH_ROWS} batches of "
                       f"{BATCH_ROWS}) after {warm_panes} warm-up panes, {args.keys} keys, hop(1s,10s); "
                       f"{threads} key-partitioned single-threaded subtasks")}


def window_checksums(torch, device, emitted):
    """Checksums of windows left on the device by handle_watermark_device: `emitted` = [(n_rows, [column pointers])]
    in the operator's output order [key, window.start, window.end, sum, avg, count, _timestamp].
    Returns [(wstart, wend, rows_out, sum of counts, wrapping sum of sums, sum of avgs)]."""
    from arroyo_b200.multi_gpu import _Ptr
    out = []
    for n, cols in emitted:
        if n == 0:
            continue
        view = lambda c: torch.as_tensor(_Ptr(cols[c], n), device=device)  # noqa: E731
        ws, we = view(1), view(2)
        out.append((int(ws[0].item()), int(we[0].item()), int(n), int(view(5).sum().item()),
                    int(view(3).sum().item()) & ((1 << 64) - 1), float(view(4).view(torch.float64).sum().item())))
    return out


OUT_COLS = ("key", "window_start", "window_end", "sum", "avg", "count", "_timestamp")  # handle_watermark_device's order
DUMP_BYTES = 64_000_000


def window_columns(torch, device, emitted):
    """Host copies of the windows of one emission left on the device (`emitted` as in window_checksums), one int64
    array per OUT_COLS name (avg: float64), rows ordered by (window start, key): the order the operator emits rows in
    follows its dictionary layout, which is not part of the result."""
    import numpy as np

    from arroyo_b200.multi_gpu import _Ptr
    parts = [[torch.as_tensor(_Ptr(cols[c], n), device=device).cpu().numpy() for c in range(len(OUT_COLS))]
             for n, cols in emitted if n]
    cols = [np.concatenate(c) for c in zip(*parts)]
    order = np.lexsort((cols[0], cols[1]))
    out = {name: c[order] for name, c in zip(OUT_COLS, cols)}
    out["avg"] = out["avg"].view(np.float64)
    return out


def dump_outputs(out_dir, cols):
    """Writes the columns as float64 .npy files under out_dir, every value exactly: a float64 column as <name>.npy, an
    int64 column (keys and nanosecond timestamps need more than float64's 53 bits) as <name>_hi.npy, its upper 32 bits
    (signed), and <name>_lo.npy, its lower 32 bits (unsigned): value = hi * 2^32 + lo.  Above DUMP_BYTES in all, every
    file keeps the same fixed, seeded sample of rows."""
    import numpy as np
    files = {}
    for name, c in cols.items():
        if c.dtype == np.float64:
            files[name] = c
        else:
            files[name + "_hi"], files[name + "_lo"] = c >> 32, c & 0xFFFFFFFF
    n = len(cols["key"])
    cap = (DUMP_BYTES - 1024 * len(files)) // (8 * len(files))  # 1 KB per file for its .npy header
    rows = np.sort(np.random.default_rng(0).choice(n, cap, replace=False)) if n > cap else slice(None)
    os.makedirs(out_dir, exist_ok=True)
    for name, c in files.items():
        np.save(os.path.join(out_dir, name + ".npy"), c[rows].astype(np.float64))


def compare_windows(got, want, min_windows):
    """got: {wstart: (wend, rows_out, counts, sums, avgs)} from the GPU run; want: the oracle's window list.
    Bit-exact rows / counts / sums (wrapping), AVG checksum within 1e-6 relative (north-star tolerance)."""
    ref = {w["wstart"]: w for w in want}
    bad, checked = [], 0
    for ws, (we, n, cnt, sm, av) in sorted(got.items()):
        w = ref.get(ws)
        if w is None:
            bad.append(f"window {ws}: not emitted by the oracle")
            continue
        checked += 1
        if (we, n, cnt, sm) != (w["wend"], w["rows_out"], w["sum_of_rows"], w["sum_of_sums"]):
            bad.append(f"window {ws}: gpu (end {we}, rows {n}, count {cnt}, sum {sm}) != oracle (end {w['wend']}, rows "
                       f"{w['rows_out']}, count {w['sum_of_rows']}, sum {w['sum_of_sums']})")
        elif abs(av - w["sum_of_avgs"]) > 1e-6 * max(abs(w["sum_of_avgs"]), 1.0):
            bad.append(f"window {ws}: avg checksum {av} vs {w['sum_of_avgs']}")
    if checked < min_windows:
        bad.append(f"only {checked} windows compared (expected at least {min_windows})")
    return {"verified": not bad, "windows_checked": checked,
            "against": "oracle/window_oracle.c (C restatement of the reference algorithm) on the same panes",
            "checks": "per window: rows out, sum COUNT(*), wrapping sum SUM(value) bit-exact; sum AVG(value) 1e-6 relative",
            **({"mismatches": bad[:8]} if bad else {})}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def build_batch_lists(torch, panes, rows_per_pane):
    """Per pane: prebuilt ctypes arrays of (key, value, ts) device pointers per 65 536-row batch, plus the
    watermark each batch triggers."""
    nb = rows_per_pane // BATCH_ROWS
    plans = []
    mins, maxs = [], []
    for (k, v, t) in panes:
        tb = t.view(nb, BATCH_ROWS)
        mins.append(tb.amin(dim=1))
        maxs.append(tb.amax(dim=1))
    mins = torch.stack(mins).cpu().numpy().reshape(-1).tolist()
    maxs = torch.stack(maxs).cpu().numpy().reshape(-1).tolist()
    wms = watermark_schedule(list(zip(mins, maxs)))
    for pi, (k, v, t) in enumerate(panes):
        segs = []  # (cols ctypes array, rows ctypes array, watermark after the run or None)
        start = 0
        for b in range(nb):
            wm = wms[pi * nb + b]
            if wm is not None or b == nb - 1:
                n = b - start + 1
                cols = (C.c_uint64 * (3 * n))()
                rows = (C.c_int64 * n)()
                for j in range(n):
                    off = (start + j) * BATCH_ROWS * 8
                    cols[3 * j + 0] = k.data_ptr() + off
                    cols[3 * j + 1] = v.data_ptr() + off
                    cols[3 * j + 2] = t.data_ptr() + off
                    rows[j] = BATCH_ROWS
                segs.append((cols, rows, wm))
                start = b + 1
        plans.append(segs)
    return plans


def bind_to_gpu_numa_node(local):
    """Pins this process to the CPUs NVML reports as local to GPU `local`, before any pinned host memory is
    allocated (first touch then places it on the GPU's NUMA node).  On this pool's two-socket hosts a process that
    lands on the other socket moves host<->device data at about 20 GB/s instead of 55.  Returns a description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return "unchanged (no overlap with the allowed CPUs)"
        os.sched_setaffinity(0, cpus)
        return f"process bound to the {len(cpus)} CPUs local to GPU {local}"
    except Exception as e:  # noqa: BLE001
        return f"unchanged ({type(e).__name__}: {e})"


def device_resident(args, torch, native, ffi, local, panes, W, K, rows, collect=False, sampler=None, last_window=None):
    """W warm-up + K timed steps over `panes` (already in HBM); CUDA events on the operator's stream.
    Returns (ms, stats delta, rows emitted, clocks, per-window checksums if `collect`).  With `collect` every emitted
    window is reduced to checksums on the device (torch kernels inside the loop): that pass verifies, it is not timed.
    A dict passed as `last_window` receives the host columns of the emission the last timed step began
    (window_columns), copied after the timed region; it is an error if that step began none, or more than one."""
    import pyarrow as pa
    device = torch.device("cuda", local)
    plans = build_batch_lists(torch, panes, rows)
    torch.cuda.synchronize()
    schema = pa.schema([("key", pa.int64()), ("value", pa.int64()), ("_timestamp", pa.timestamp("ns"))])
    flags = ffi.FLAG_PROFILE | op_flags(args)
    stream = torch.cuda.current_stream().cuda_stream
    op = native.SlidingAggregatingWindowFunc(window_config(), input_schema=schema, device=local, stream=stream,
                                             flags=flags, expected_keys=args.keys, chunk_log2=args.chunk_log2)
    rows_out = 0
    sums = {}
    last_step, last, n_last = W + K - 1, [], 0  # the last timed step's emission and how many it began

    outstanding = None  # the step that began the emission still to be polled

    def gather():
        # the windows of the outstanding emission (arroyo_b200_op_handle_watermark_device_poll)
        nonlocal rows_out, outstanding, last, n_last
        if outstanding is None:
            return
        by, outstanding = outstanding, None
        emitted = op.handle_watermark_device_poll()
        if by == last_step:
            last, n_last = emitted, n_last + 1
        for n, _ in emitted:
            rows_out += n
        if collect:
            for ws, we, n, cnt, sm, av in window_checksums(torch, device, emitted):
                sums[ws] = (we, n, cnt, sm, av)

    def step(p):
        # handle_watermark as the begin / poll pair: the emission is enqueued, the next batches are handed over and
        # submitted behind it, and only then are the emitted windows' row counts read -- the device never idles while
        # the host goes round (with `--sync-emit`: the blocking call, one round trip more per step)
        nonlocal rows_out, outstanding
        for cols, nrows, wm in plans[p]:
            op.process_device_batches(cols, nrows, 3)
            if wm is None:
                continue
            if args.sync_emit:
                outstanding = p
                op.handle_watermark_device_begin(wm)
                gather()
                continue
            op.submit()
            gather()
            op.handle_watermark_device_begin(wm)
            outstanding = p

    if sampler is None:
        sampler = ClockSampler(local)
        if not collect:
            sampler.start()
    for p in range(W):
        step(p)
    gather()
    op.flush()
    torch.cuda.synchronize()
    st0 = op.stats()
    rows_out = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.begin()
    e0.record()
    for p in range(W, W + K):
        step(p)
    gather()
    op.flush()
    e1.record()
    torch.cuda.synchronize()
    sampler.end()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if not collect else None
    if last_window is not None:
        # flush() emits nothing: the buffers still hold the last emission until the operator's next one (which is also
        # why only one emission of the step can be read here)
        if n_last != 1 or not any(n for n, _ in last):
            raise RuntimeError(f"the last timed step began {n_last} emissions (rows: {[n for n, _ in last]}); "
                               "--dump-outputs writes the windows of its one emission")
        last_window.update(window_columns(torch, device, last))
    st1 = op.stats()
    op.close()
    del plans
    torch.cuda.empty_cache()
    return ms, {k: st1[k] - st0[k] for k in st1}, rows_out, clocks, sums


def run_ours(args):
    import torch
    import torch.distributed as dist

    import arroyo_b200 as ab
    from arroyo_b200 import ffi, operators as native

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    all_cpus = os.sched_getaffinity(0)
    args.numa = "not bound" if args.no_numa_bind else bind_to_gpu_numa_node(local)
    if world > 1:
        # whole-job watchdog: a rank that sits in one phase (communicator set-up, a collective whose peer never
        # arrives ...) for seven minutes says where, dumps its threads' stacks and exits, instead of hanging silently
        from arroyo_b200.multi_gpu import _Watchdog
        args._dog = _Watchdog(rank, f"bench.py at {world} GPUs", limit_s=420.0)
        args._dog.beat("init_process_group")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        args._dog.beat("process group up")
    if ffi.load().arroyo_b200_device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: arroyo_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    # one explicit CUDA stream for torch and the operator: the CUDA events below are recorded on the stream the
    # kernels are launched on (a stream handle of 0 would make the operator create a private stream)
    # (high priority: at N > 1 the exchange and the owner stage run on it while the local stage's ingest kernels
    # fill the GPU from another stream)
    torch.cuda.set_stream(torch.cuda.Stream(device=device, priority=-1))
    if world > 1:
        from arroyo_b200 import multi_gpu
        return multi_gpu.bench(args, torch, dist, rank, world, local, all_cpus)

    W, K = steady_warmup(args.warmup), args.steps
    rows = args.rows_per_pane
    assert rows % BATCH_ROWS == 0
    gen_pane = make_generator(torch, device, rows, args.keys, args.dist, 42 + rank, args.keyspace)
    panes = [gen_pane(p) for p in range(W + K)]
    last_window = {} if args.dump_outputs else None
    ms, d, rows_out, clocks, _ = device_resident(args, torch, native, ffi, local, panes, W, K, rows,
                                                 last_window=last_window)
    del panes
    if last_window is not None:
        dump_outputs(args.dump_outputs, last_window)

    value = K * rows / (ms * 1e-3)
    peak, peak_kind = measured_peak()
    ingest_gbs = 24.0 * d["ingest_rows_timed"] / (d["ingest_ms"] * 1e-3) / 1e9 if d["ingest_ms"] else None
    emit_share = d["emit_ms"] / ms if ms else None
    step_bytes = 24.0 * rows + 72.0 * args.keys + 48.0 * (rows_out / max(K, 1))
    traffic = ncu_traffic()
    alg_per_launch = 24.0 * d["ingest_rows_timed"] / max(d["ingest_launches"], 1)
    roof = {"bound": "hbm", "kernel": (traffic or {}).get("kernel", "ingest"),
            "achieved": round(ingest_gbs, 1) if ingest_gbs else None,
            "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
            "frac": round(ingest_gbs / peak, 4) if ingest_gbs else None,
            # DRAM bytes of the ncu capture scaled to this run's launch size (the capture's own launch is recorded
            # beside it), so `traffic` and `algorithmic_bytes_per_launch` describe the same launch
            "traffic": (round(traffic["dram_bytes_per_row"] * d["ingest_rows_timed"] / max(d["ingest_launches"], 1))
                        if traffic and traffic.get("dram_bytes_per_row") else None),
            "traffic_source": (traffic or {}).get("source"),
            "algorithmic_bytes_per_launch": alg_per_launch,
            "ingest_ms_per_step": d["ingest_ms"] / K, "emit_ms_per_step": d["emit_ms"] / K,
            "ingest_share_of_step": round(d["ingest_ms"] / ms, 3), "emit_share_of_step": round(emit_share, 3),
            "pipeline_frac": round(step_bytes * K / (ms * 1e-3) / 1e9 / peak, 4),
            "host_process_ms_per_step": round(d["host_process_ms"] / K, 4),
            "host_watermark_ms_per_step": round(d["host_watermark_ms"] / K, 4)}

    out = {"metric": "rows/sec sliding-window SUM (1M keys)", "value": value, "unit": "rows/s", "n_gpus": 1,
           "steps": K, "warmup": W, "warmup_requested": args.warmup, "ms_per_step": ms / K, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
           "config": workload_config(args, 1),
           "impl": {"emission": "remerge" if args.remerge else "running add/evict",
                    "avg": "f64 accumulator" if args.avg_f64 else "exact integer sum (guarded)",
                    "combine": not args.no_combine, "numa": args.numa,
                    "ingest": ("one pass: probe + one RED per accumulator per row" if args.one_pass else
                               "two passes: radix partition by dictionary bucket, per-bucket aggregation in shared memory"),
                    "warmup_note": "warm-up = max(--warmup, width/slide + 3) panes: the timed steps see the steady state"},
           "rows_out_per_step": rows_out / max(K, 1), "gpu_launches": int(d["kernel_launches"]),
           "roofline": roof, "clocks": clocks}

    # ---- e2e: host Arrow batches in, host Arrow batches out, through the reference-facing call ----
    if not args.skip_e2e:
        out["e2e"] = run_e2e(args, torch, device, local, gen_pane)
    if not args.skip_cpu:
        os.sched_setaffinity(0, all_cpus)  # the CPU baseline gets every host core again
        cpu = run_cpu(torch, args, device, budget_s=25.0, warm_panes=11, timed_panes=3)
        out["cpu_baseline"] = {"value": cpu["rows_per_s"], "unit": "rows/s", "cores": cpu["threads"], "kind": "port",
                               "sample": cpu["sample"]}
        # ---- verify: the GPU operator over the very panes the oracle just consumed, window by window ----
        vp = [sample_pane(torch, device, gen_pane(p), cpu["rows_per_step"]) for p in range(cpu["panes"])]
        _, _, _, _, sums = device_resident(args, torch, native, ffi, local, vp, cpu["panes"], 0, cpu["rows_per_step"],
                                           collect=True)
        out["verify"] = compare_windows(sums, cpu["windows"], min_windows=cpu["panes"] - 4)
        out["verify"]["rows_per_pane"] = cpu["rows_per_step"]
        out["verify"]["panes"] = cpu["panes"]
        out["verified"] = out["verify"]["verified"]
    print(json.dumps(out), flush=True)
    if out.get("verified") is False:
        sys.exit("bench.py: GPU windows differ from the oracle's -- see the verify block of the line above")


def host_feed(torch, gen_pane, pane_ids, rows, pinned=True):
    """Host copies of the given panes as Arrow batches of BATCH_ROWS rows (zero copy: the Arrow buffers *are* the
    host memory: page-locked by default, what a shim gets from arroyo_b200_host_alloc; `pinned=False` = ordinary
    pageable allocations, what arrow-rs hands out by itself) and the watermark each batch triggers."""
    import pyarrow as pa
    nb = rows // BATCH_ROWS
    host_pool = {}
    host = []
    for p in pane_ids:
        k, v, t = gen_pane(p)
        if p % POOL not in host_pool:
            hk = torch.empty(rows, dtype=torch.int64, pin_memory=pinned)
            hv = torch.empty(rows, dtype=torch.int64, pin_memory=pinned)
            hk.copy_(k)
            hv.copy_(v)
            host_pool[p % POOL] = (hk, hv)
        ht = torch.empty(rows, dtype=torch.int64, pin_memory=pinned)
        ht.copy_(t)
        host.append([host_pool[p % POOL][0], host_pool[p % POOL][1], ht])
    torch.cuda.synchronize()
    ts_type = pa.timestamp("ns")

    def arrow_batch(cols, b):
        arrs = []
        for ci, h in enumerate(cols):
            a = h.numpy()[b * BATCH_ROWS:(b + 1) * BATCH_ROWS]
            arrs.append(pa.Array.from_buffers(ts_type if ci == 2 else pa.int64(), BATCH_ROWS, [None, pa.py_buffer(a)]))
        return pa.RecordBatch.from_arrays(arrs, names=["key", "value", "_timestamp"])

    batches = [[arrow_batch(cols, b) for b in range(nb)] for cols in host]
    mm = []
    for cols in host:
        t = cols[2].view(nb, BATCH_ROWS)
        mm += list(zip(t.amin(dim=1).tolist(), t.amax(dim=1).tolist()))
    return batches, watermark_schedule(mm), host


def run_e2e(args, torch, device, local, gen_pane):
    import pyarrow as pa

    import arroyo_b200 as ab
    from arroyo_b200 import ffi, operators as native
    K = args.e2e_steps or min(args.steps, 10)
    W = steady_warmup(0)
    rows = args.rows_per_pane
    nb = rows // BATCH_ROWS
    batches, wms, _keep = host_feed(torch, gen_pane, range(W + K), rows)
    host_kind = "pinned"

    def trial():
        """One fresh operator over the same pinned host batches: W warm-up panes, K timed panes."""
        op = native.SlidingAggregatingWindowFunc(window_config(), device=local, expected_keys=args.keys,
                                                 flags=op_flags(args))
        ctx = ab.OperatorContext(1)
        col = ab.Collector()
        d2h = 0
        outstanding = False  # an emission whose windows are still on their way to the host

        def collect(block):
            """The shim's handle_future_result: take the windows of the outstanding emission (then it would forward the
            watermark it held back)."""
            nonlocal d2h, outstanding
            if not outstanding or not op.handle_watermark_poll(col, block=block):
                return
            outstanding = False
            for rb in col.batches:
                d2h += rb.num_rows * 48
            col.batches.clear()

        def step(p):
            nonlocal d2h, outstanding
            for b in range(nb):
                op.process_batch(batches[p][b], ctx, col)
                wm = wms[p * nb + b]
                if wm is not None:
                    ctx.watermarks.set(0, wm)
                    if args.sync_emit:
                        op.handle_watermark(wm, ctx, col)
                        for rb in col.batches:
                            d2h += rb.num_rows * 48
                        col.batches.clear()
                    else:
                        collect(block=True)  # windows leave in order: the previous emission first
                        outstanding = op.handle_watermark_begin(wm, ctx)
                elif outstanding and b % 8 == 0:
                    collect(block=False)  # the run loop polls the future between batches

        if args.e2e_host == "library":
            # the subtask run loop in compiled code: one arroyo_b200_op_run_batches call per pane's worth of queued
            # batches.  Exporting a batch builds Arrow C descriptors only (no buffer is touched), so it is done ahead.
            import ctypes as C
            exported = [native.ExportedBatches(batches[p]) for p in range(W + K)]
            wm_arr = []
            for p in range(W + K):
                a = (C.c_int64 * nb)(*[ffi.NO_WATERMARK if wms[p * nb + b] is None else wms[p * nb + b] for b in range(nb)])
                wm_arr.append(a)

            def step(p):  # noqa: F811
                nonlocal d2h
                op.run_batches(exported[p], wm_arr[p], col, async_emit=not args.sync_emit)
                for rb in col.batches:
                    d2h += rb.num_rows * 48
                col.batches.clear()

            def collect(block):  # noqa: F811
                nonlocal d2h
                op.handle_watermark_poll(col, block=block)
                for rb in col.batches:
                    d2h += rb.num_rows * 48
                col.batches.clear()

        for p in range(W):
            step(p)
        collect(block=True)
        op.flush()
        torch.cuda.synchronize()
        d2h = 0
        st0 = op.stats()
        t0 = time.perf_counter()
        for p in range(W, W + K):
            step(p)
        collect(block=True)
        op.flush()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        st1 = op.stats()
        op.close()
        how = ("arroyo_b200_op_handle_watermark" if args.sync_emit else
               "arroyo_b200_op_handle_watermark_begin / _poll (windows copied back while the next batches are copied in)")
        loop = ("arroyo_b200_op_run_batches (run loop inside the library)" if args.e2e_host == "library" else
                "arroyo_b200_op_process_batch per batch from Python")
        return {"value": K * rows / dt, "unit": "rows/s", "host_buffers": host_kind, "h2d_bytes_per_step": rows * 24,
                "d2h_bytes_per_step": d2h // max(K, 1), "steps": K, "ms_per_step": 1e3 * dt / K,
                "host_process_ms_per_step": round((st1["host_process_ms"] - st0["host_process_ms"]) / K, 3),
                "host_watermark_ms_per_step": round((st1["host_watermark_ms"] - st0["host_watermark_ms"]) / K, 3),
                "path": f"pinned host Arrow batches -> {loop} -> {how} -> host Arrow windows"}

    # The host link is shared with the box's other tenants (a neighbour's copies can halve a 100 ms measurement),
    # so the pass is repeated: the median trial is reported, every trial is listed.
    n_trials = max(1, args.e2e_trials)
    results = [trial() for _ in range(n_trials)]
    results.sort(key=lambda r: r["value"])
    out = dict(results[len(results) // 2])
    out["trials"] = [round(r["value"]) for r in results]
    out["trials_note"] = f"median of {n_trials} passes (fresh operator each, same pinned host batches)"
    out["host_buffers_note"] = ("Arrow buffers are page-locked (cudaHostAlloc; a shim allocates its batch buffers with "
                                "arroyo_b200_host_alloc).  `pageable` = the same pass over ordinary pageable buffers, "
                                "which the driver stages through its own bounce buffers")
    if not args.skip_pageable:
        # arrow-rs allocates pageable memory unless told otherwise: the same run over pageable buffers, one pass
        del batches, _keep
        K = min(K, 5)
        batches, wms, _keep = host_feed(torch, gen_pane, range(W + K), rows, pinned=False)
        host_kind = "pageable"
        pg = trial()
        out["pageable"] = {"value": pg["value"], "unit": "rows/s", "steps": K, "ms_per_step": pg["ms_per_step"]}
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  The Rust
    reference cannot be built in this image (no rustc/cargo, DataFusion/arrow-rs not vendored), so this is
    the C port of its algorithm (oracle/window_oracle.c), pinned by the reference's golden vectors.
    At --gpus N the subtasks consume the union of the N source shards (the same stream the N GPUs consume)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else torch.device("cpu")
    world = max(1, args.gpus)
    W, K = steady_warmup(args.warmup), args.steps
    cpu = run_cpu(torch, args, device, budget_s=150.0, warm_panes=W, timed_panes=K, seeds=tuple(42 + r for r in range(world)))
    line = {"impl": "reference", "metric": "rows/sec sliding-window SUM (1M keys)", "value": cpu["rows_per_s"],
            "unit": "rows/s", "n_gpus": args.gpus, "steps": cpu["steps"], "warmup": W, "warmup_requested": args.warmup,
            "ms_per_step": cpu["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": workload_config(args, world),
            "cpu_baseline": {"value": cpu["rows_per_s"], "unit": "rows/s", "cores": cpu["threads"], "kind": "port",
                             "sample": cpu["sample"]},
            "e2e": {"value": cpu["rows_per_s"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_reference_workload(args):
    """--impl reference --workload join | session: the C restatement of the operator on the host cores (rank 0)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import bench_workloads as BW
    world = max(1, args.gpus)
    if args.workload == "join":
        v, cores, sample = BW.cpu_join(1 << args.join_persons_log2, 1 << args.join_auctions_log2, world, budget_s=60.0)
        metric = "input rows/sec windowed hash-join (Nexmark q8 shape)"
    else:
        v, cores, sample = BW.cpu_session(args.session_keys, 1 << args.session_rows_log2, world, budget_s=60.0)
        metric = "rows/sec session-window aggregate (5 s gap)"
    print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": "rows/s", "n_gpus": args.gpus,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                      "config": {"workload": args.workload, "n_gpus": world},
                      "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample},
                      "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}), flush=True)


def main():
    args = parse()
    if args.workload != "sliding":
        if args.impl == "reference":
            run_reference_workload(args)
        else:
            import bench_workloads
            bench_workloads.run(args, sys.modules[__name__])
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
