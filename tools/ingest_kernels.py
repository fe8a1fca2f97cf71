"""Per-kernel split of the benchmark's device-resident steps: runs bench.py's steady-state loop (bench.make_generator +
bench.device_resident, same arguments as bench.py) under torch.profiler with CUDA activities and prints, as one JSON
line, the mean microseconds per launch of the sliding window's kernels, with the card's name and power limit.

    python tools/ingest_kernels.py --steps 20 --warmup 12

The profiler slows the host, not the kernels: take step times from bench.py, per-kernel times from here.
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KERNELS = ("part_kernel", "agg_kernel", "emit_kernel", "pane_init_kernel")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, limit = (x.strip() for x in out[0].split(","))
        return name, limit
    except Exception as e:  # noqa: BLE001 -- the table is still worth printing without it
        return None, f"unavailable: {e}"


def main():
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench as B
    from arroyo_b200 import ffi, operators as native

    args = B.parse()
    if ffi.load().arroyo_b200_device_count() < 1:
        raise RuntimeError("ingest_kernels.py needs a CUDA device")
    torch.cuda.set_device(0)
    device = torch.device("cuda", 0)
    torch.cuda.set_stream(torch.cuda.Stream(device=device, priority=-1))
    W, K = B.steady_warmup(args.warmup), args.steps
    rows = args.rows_per_pane
    gen = B.make_generator(torch, device, rows, args.keys, args.dist, 42, args.keyspace)
    panes = [gen(p) for p in range(W + K)]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ms = B.device_resident(args, torch, native, ffi, 0, panes, W, K, rows)[0]
        torch.cuda.synchronize()
    per = {k: [0, 0.0] for k in KERNELS}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                per[k][0] += ev.count
                per[k][1] += ev.self_device_time_total
    name, limit = card()
    res = {"card": name, "power_limit": limit, "steps": W + K, "rows_per_pane": rows, "dist": args.dist,
           "keyspace": args.keyspace, "timed_ms_per_step_under_profiler": ms / K if K else None,
           "kernels": {k: {"launches": n, "mean_us": round(t / n, 2) if n else None, "us_per_step": round(t / (W + K), 2)}
                       for k, (n, t) in per.items()}}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
