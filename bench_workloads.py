"""`bench.py --workload join | session`: BASELINE configs[3] and configs[4] as bench lines at N >= 1 GPUs.

    join     Nexmark-q8-shaped windowed hash join: per 30-s tumbling window every GPU's source shard delivers
             2^21 persons and 2^23 auctions (one instant per window, like the rows a tumbling aggregate hands on);
             both inputs cross a key-hash Shuffle edge (person id / seller), the owner's InstantJoin joins them
             when the min-merged watermark of its two inputs releases the window.
    session  session-window aggregate, gap 5 s, 10 M keys per GPU: every GPU's shard delivers 2^22 rows per second of
             event time, raw rows cross the Shuffle edge by key, the owner's SessionAggregatingWindowFunc aggregates.

Weak scaling (per-GPU input fixed).  The Shuffle edge at N > 1 is the library's own round (csrc/exchange.cu: partition +
control all-gather + grouped ncclSend / ncclRecv), every sender's block reaches the owner's operator as its own batch (the
reference's receiver sees one batch per sender; session results depend on what shares a batch).  At N = 1 the edge is the
identity (one subtask: the reference's collector forwards without repartitioning).

One JSON line like bench.py's: `value` = input rows/s of the whole job, device-resident, CUDA events, max over ranks;
`verified` = the same N-GPU plan at a size the numpy oracle finishes in seconds gives the oracle's result (checksums over
every output column, summed over the owners); `cpu_baseline` = the C restatement of the reference operator
(oracle/join_oracle.c, oracle/session_oracle.c) on a bounded sample, one single-threaded subtask per key partition on the
host's cores -- the reference's dataflow shape.  (Only the two functions named cpu_* / verify_* touch oracle/.)
"""
import ctypes as C
import json
import os
import sys
import time

S = 1_000_000_000
T0 = 1_700_000_000 * S
MULT = (0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F, 0x165667B19E3779F9, 0x27D4EB2F165667C5, 0x85EBCA77C2B2AE63,
        0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53)


def _i64(x):
    x &= (1 << 64) - 1
    return x - (1 << 64) if x >> 63 else x


class Edge:
    """One Shuffle edge carrying raw rows.  round(cols, n, wm) -> ([(col pointers, rows) per sender], effective watermark
    or None).  The returned blocks stay valid for two rounds."""

    def __init__(self, torch, dist, rank, world, local, stream, n_cols, key_col, max_rows):
        self.world = world
        self.ex = None
        self.last = None
        if world > 1:
            from arroyo_b200.native_exchange import NativeExchange
            self.ex = NativeExchange(torch, dist, rank, world, local, stream, n_cols, key_col, max_rows, 2 * max_rows)

    def round(self, cols, n, wm):
        if self.ex is None:
            eff = wm if (wm is not None and wm != self.last) else None
            self.last = wm if wm is not None else self.last
            return ([(cols, n)] if n else []), eff
        got, eff, _ = self.ex.round_packed(cols, None, n, wm)
        return got, eff

    def close(self):
        if self.ex is not None:
            self.ex.close()


def _checksum(torch, ptr_cols, n, device):
    """(rows, wrapping sum over rows of sum_c col_c * MULT[c]) of one device batch."""
    from arroyo_b200.multi_gpu import _Ptr
    acc = torch.zeros((), dtype=torch.int64, device=device)
    for c, p in enumerate(ptr_cols):
        col = torch.as_tensor(_Ptr(p, n), device=device)
        acc = acc + (col * _i64(MULT[c % len(MULT)])).sum()
    return n, acc


def _np_checksum(np, cols):
    tot = 0
    for c, col in enumerate(cols):
        a = np.ascontiguousarray(col)
        if a.dtype != np.int64:
            a = a.view(np.int64) if a.dtype.itemsize == 8 else a.astype(np.int64)
        with np.errstate(over="ignore"):
            tot += int((a * np.int64(_i64(MULT[c % len(MULT)]))).sum(dtype=np.int64))
    return _i64(tot)


# ---------------------------------------------------------------------------------------------------------------
# join
# ---------------------------------------------------------------------------------------------------------------
def _join_inputs(torch, device, rank, world, n_p, n_a, seed):
    g = torch.Generator(device=device)
    g.manual_seed(seed + rank)
    pid = torch.randperm(n_p, device=device, generator=g).to(torch.int64) + (1000 + rank * n_p)
    name = torch.randint(0, 10**6, (n_p,), device=device, generator=g, dtype=torch.int64)
    seller = torch.randint(0, world * n_p, (n_a,), device=device, generator=g, dtype=torch.int64) + 1000
    auction = torch.arange(n_a, device=device, dtype=torch.int64) + rank * n_a
    reserve = torch.randint(1, 10**5, (n_a,), device=device, generator=g, dtype=torch.int64)
    return pid, name, seller, auction, reserve


def _run_join(torch, dist, rank, world, local, device, n_p, n_a, warm, steps, seed, collect=False, sampler=None):
    import pyarrow as pa

    import arroyo_b200 as ab
    from arroyo_b200 import ffi, operators as native
    from arroyo_b200.context import clamp_watermark
    stream = torch.cuda.current_stream().cuda_stream
    W30 = 30 * S
    l_schema = pa.schema([("id", pa.int64()), ("name_code", pa.int64()), ("_timestamp", pa.timestamp("ns"))])
    r_schema = pa.schema([("seller", pa.int64()), ("auction", pa.int64()), ("reserve", pa.int64()),
                          ("_timestamp", pa.timestamp("ns"))])
    jop = native.InstantJoin(ab.JoinConfig(left_on=["id"], right_on=["seller"], join_type="inner"), left_schema=l_schema,
                             right_schema=r_schema, device=local, stream=stream)
    el = Edge(torch, dist, rank, world, local, stream, 3, 0, n_p)
    er = Edge(torch, dist, rank, world, local, stream, 4, 0, n_a)
    pid, name, seller, auction, reserve = _join_inputs(torch, device, rank, world, n_p, n_a, seed)
    tl = [torch.empty(n_p, device=device, dtype=torch.int64) for _ in range(2)]
    tr = [torch.empty(n_a, device=device, dtype=torch.int64) for _ in range(2)]
    holder = ab.WatermarkHolder(2)
    lib, h = jop._lib, jop._h
    outb = (ffi.DeviceBatch * 8)()
    rows_out = 0
    sums = []
    applied = None

    def feed(side, got, n_cols):
        for cols, n in got:
            arr = (C.c_uint64 * n_cols)(*cols)
            native._check(lib, h, lib.arroyo_b200_op_process_device_batch(h, side, 2, arr, n_cols, n))

    def step(w):
        nonlocal rows_out, applied
        ts = T0 + (w + 1) * W30 - 1
        a, b = tl[w & 1], tr[w & 1]
        a.fill_(ts)
        b.fill_(ts)
        got, eff = el.round([pid.data_ptr(), name.data_ptr(), a.data_ptr()], n_p, ts + 1)
        feed(0, got, 3)
        if eff is not None:
            holder.set(0, eff)
        got, eff = er.round([seller.data_ptr(), auction.data_ptr(), reserve.data_ptr(), b.data_ptr()], n_a, ts + 1)
        feed(1, got, 4)
        if eff is not None:
            holder.set(1, eff)
        cur = holder.last_present_watermark
        if cur is not None and cur != applied:
            applied = cur
            n = C.c_int64(0)
            native._check(lib, h, lib.arroyo_b200_op_handle_watermark_device(h, clamp_watermark(cur), outb, 8, C.byref(n)))
            for i in range(n.value):
                rows_out += outb[i].n_rows
                if collect:
                    sums.append(_checksum(torch, [outb[i].cols[c] for c in range(outb[i].n_cols)], outb[i].n_rows, device))

    if sampler is not None:
        sampler.start()  # after the set-up (operators, NCCL communicators), right before the warm-up
    for w in range(warm):
        step(w)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    rows_out = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler is not None:
        sampler.begin()
    e0.record()
    for w in range(warm, warm + steps):
        step(w)
    e1.record()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.end()
    ms = e0.elapsed_time(e1) if steps else 0.0
    launches = jop.stats()["kernel_launches"]
    jop.close()
    el.close()
    er.close()
    return ms, rows_out, sums, launches


def verify_join(torch, dist, rank, world, local, device, seed=7):
    """The N-GPU plan at 2^12 persons x 2^14 auctions per GPU and window against the numpy oracle's InstantJoin over the
    union of the shards (an inner join's result does not depend on who owns a key)."""
    n_p, n_a, windows = 1 << 12, 1 << 14, 3
    _, rows, sums, _ = _run_join(torch, dist, rank, world, local, device, n_p, n_a, windows, 0, seed, collect=True)
    t = torch.tensor([sum(n for n, _ in sums), 0], dtype=torch.int64, device=device)
    for _, s in sums:
        t[1] += s
    if dist is not None:
        dist.all_reduce(t)
    got = (int(t[0].item()), int(t[1].item()))
    if rank != 0:
        return None
    import numpy as np

    from oracle import arroyo_oracle as O
    ins = [[x.cpu().numpy() for x in _join_inputs(torch, device, r, world, n_p, n_a, seed)] for r in range(world)]
    join = O.InstantJoin(O.JoinConfig(left_on=["id"], right_on=["seller"], join_type="inner"))
    ctx, out = O.OperatorContext(2), O.Collector()
    want_rows, want_sum = 0, 0
    for w in range(windows):
        ts = T0 + (w + 1) * 30 * S - 1
        for pid, name, seller, auction, reserve in ins:
            join.process_batch_index(0, 2, O.Batch({"id": pid, "name_code": name,
                                                    O.TIMESTAMP: np.full(n_p, ts, dtype=np.int64)}), ctx, out)
            join.process_batch_index(1, 2, O.Batch({"seller": seller, "auction": auction, "reserve": reserve,
                                                    O.TIMESTAMP: np.full(n_a, ts, dtype=np.int64)}), ctx, out)
        for side in (0, 1):
            ctx.watermarks.set(side, ts + 1)
        join.handle_watermark(ts + 1, ctx, out)
    names = ["id", "name_code", "seller", "auction", "reserve", O.TIMESTAMP]
    for b in out.batches:
        want_rows += b.num_rows
        want_sum = _i64(want_sum + _np_checksum(np, [b[c] for c in names]))
    ok = got == (want_rows, want_sum)
    return {"verified": ok, "rows_out": got[0], "expected_rows_out": want_rows,
            "against": "oracle/arroyo_oracle.py InstantJoin on the union of the shards",
            "checks": "joined rows and a wrapping checksum over every output column, summed over the owners",
            "size": f"{n_p} persons x {n_a} auctions per GPU and window, {windows} windows"}


def cpu_join(n_p, n_a, world, budget_s=20.0):
    """oracle/join_oracle.c on the union of `world` shards of one window, key-partitioned over P single-threaded
    subtasks (threads: the C calls release the GIL).  A bounded sample: the shard size shrinks until a window fits the
    budget.  Returns (input rows/s, threads, sample description)."""
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np

    from oracle import arroyo_oracle as O, c_oracle
    P = max(1, min(os.cpu_count() or 1, 64))
    while True:
        rng = np.random.default_rng(1)
        tp, ta = n_p * world, n_a * world
        pid = rng.permutation(tp).astype(np.int64) + 1000
        name = rng.integers(0, 10**6, tp, dtype=np.int64)
        seller = rng.integers(0, tp, ta, dtype=np.int64) + 1000
        auction = np.arange(ta, dtype=np.int64)
        reserve = rng.integers(1, 10**5, ta, dtype=np.int64)
        lp, rp = pid % P, seller % P
        parts = [(pid[lp == q], name[lp == q], seller[rp == q], auction[rp == q], reserve[rp == q]) for q in range(P)]

        def work(part, windows=2):
            p_, n_, s_, a_, r_ = part
            join = c_oracle.InstantJoin(O.JoinConfig(left_on=["id"], right_on=["seller"], join_type="inner"))
            ctx, out = O.OperatorContext(2), O.Collector()
            t0 = None
            for w in range(windows + 1):
                if w == 1:
                    t0 = time.perf_counter()  # the first window warms the allocations up
                ts = T0 + (w + 1) * 30 * S - 1
                join.process_batch_index(0, 2, O.Batch({"id": p_, "name_code": n_, O.TIMESTAMP: np.full(len(p_), ts, dtype=np.int64)}), ctx, out)
                join.process_batch_index(1, 2, O.Batch({"seller": s_, "auction": a_, "reserve": r_,
                                                        O.TIMESTAMP: np.full(len(s_), ts, dtype=np.int64)}), ctx, out)
                for side in (0, 1):
                    ctx.watermarks.set(side, ts + 1)
                join.handle_watermark(ts + 1, ctx, out)
                out.batches.clear()
            return (time.perf_counter() - t0) / windows

        t0 = time.perf_counter()
        with ThreadPoolExecutor(P) as pool:
            per_window = max(pool.map(work, parts))
        if time.perf_counter() - t0 <= budget_s or n_a <= (1 << 16):
            return (tp + ta) / per_window, P, f"2 windows of {tp} persons x {ta} auctions over {P} key-partitioned subtasks"
        n_p //= 4
        n_a //= 4


# ---------------------------------------------------------------------------------------------------------------
# session
# ---------------------------------------------------------------------------------------------------------------
def _session_step_inputs(torch, device, rank, n_keys, srows, n_steps, seed):
    g = torch.Generator(device=device)
    g.manual_seed(seed + rank)
    keys = [torch.randint(0, n_keys, (srows,), device=device, generator=g, dtype=torch.int64) * 7919 + rank
            for _ in range(n_steps)]
    val = torch.randint(0, 10**6, (srows,), device=device, generator=g, dtype=torch.int64)
    offs = torch.sort(torch.randint(0, S, (srows,), device=device, generator=g, dtype=torch.int64)).values
    return keys, val, offs


def _session_cfg(mod):
    return mod.SessionConfig(gap=5 * S, key_names=["key"], aggs=[mod.Agg("sum", "value", "sum"), mod.Agg("count", None, "n")],
                             window_index=1)


def _run_session(torch, dist, rank, world, local, device, n_keys, srows, warm, steps, seed, collect=False, final=False,
                 split=1, sampler=None):
    import pyarrow as pa

    import arroyo_b200 as ab
    from arroyo_b200 import operators as native
    stream = torch.cuda.current_stream().cuda_stream
    schema = pa.schema([("key", pa.int64()), ("value", pa.int64()), ("_timestamp", pa.timestamp("ns"))])
    sop = native.SessionAggregatingWindowFunc(_session_cfg(ab), input_schema=schema, device=local, stream=stream,
                                              expected_keys=n_keys)
    edge = Edge(torch, dist, rank, world, local, stream, 3, 0, srows)
    keys, val, offs = _session_step_inputs(torch, device, rank, n_keys, srows, warm + steps, seed)
    tsb = [torch.empty(srows, device=device, dtype=torch.int64) for _ in range(2)]
    rows_out = 0
    sums = []
    keep = []

    def emit(wm):
        nonlocal rows_out
        for n, cols in sop.handle_watermark_device(wm):
            rows_out += n
            if collect:
                sums.append(_checksum(torch, cols, n, device))

    def step(p):
        ts = tsb[p & 1]
        torch.add(offs, T0 + p * S, out=ts)
        got, eff = edge.round([keys[p].data_ptr(), val.data_ptr(), ts.data_ptr()], srows, T0 + p * S - S)
        if split > 1 and world == 1:
            # measurement knob: what an owner behind `split` senders sees -- `split` batches per step that cover the same
            # second (rows j, j + split, j + 2 split, ... of the step)
            parts = [(keys[p][j::split].contiguous(), val[j::split].contiguous(), ts[j::split].contiguous()) for j in range(split)]
            keep.append(parts)
            del keep[:-2]
            got = [([k.data_ptr(), v.data_ptr(), t.data_ptr()], k.numel()) for k, v, t in parts]
        for cols, n in got:  # one batch per sender, in sender order
            sop.process_device_batch(cols, n)
        if eff is not None:
            emit(eff)

    if sampler is not None:
        sampler.start()  # after the set-up (operator, NCCL communicator), right before the warm-up
    for p in range(warm):
        step(p)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    rows_out = 0 if not collect else rows_out
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler is not None:
        sampler.begin()
    e0.record()
    for p in range(warm, warm + steps):
        step(p)
    e1.record()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.end()
    ms = e0.elapsed_time(e1) if steps else 0.0
    if final:  # end of data: every open session leaves
        got, eff = edge.round(None, 0, ab.FINAL_WATERMARK)
        if eff is not None:
            emit(eff)
    launches = sop.stats()["kernel_launches"]
    sop.close()
    edge.close()
    return ms, rows_out, sums, launches


def verify_session(torch, dist, rank, world, local, device, seed=11):
    """The N-GPU plan on 14 one-second steps of 4096 rows per GPU (20 000 keys per GPU) plus the end-of-data watermark,
    against a single-process simulation of the same world x world topology with the numpy oracle's session operator
    (every sender's block is its own batch, senders in rank order, watermarks min-merged per owner)."""
    n_keys, srows, n_steps = 20_000, 4096, 14  # a key sees a row every ~5 steps: gaps on both sides of the 5-s session gap
    _, _, sums, _ = _run_session(torch, dist, rank, world, local, device, n_keys, srows, n_steps, 0, seed, collect=True,
                                 final=True)
    t = torch.tensor([sum(n for n, _ in sums), 0], dtype=torch.int64, device=device)
    for _, s in sums:
        t[1] += s
    if dist is not None:
        dist.all_reduce(t)
    got = (int(t[0].item()), int(t[1].item()))
    if rank != 0:
        return None
    import numpy as np

    from oracle import arroyo_oracle as O
    shards = []
    for r in range(world):
        keys, val, offs = _session_step_inputs(torch, device, r, n_keys, srows, n_steps, seed)
        shards.append(([k.cpu().numpy() for k in keys], val.cpu().numpy(), offs.cpu().numpy()))
    ops = [O.SessionAggregatingWindowFunc(_session_cfg(O)) for _ in range(world)]
    ctxs = [O.OperatorContext(world) for _ in range(world)]
    outs = [O.Collector() for _ in range(world)]
    for p in range(n_steps + 1):
        wms = []
        for s in range(world):
            if p < n_steps:
                keys, val, offs = shards[s]
                b = O.Batch({"key": keys[p], "value": val, O.TIMESTAMP: offs + (T0 + p * S)})
                for d, sb in (O.repartition(b, ["key"], world) if world > 1 else [(0, b)]):
                    ops[d].process_batch(sb, ctxs[d], outs[d])
                wms.append(T0 + p * S - S)
            else:
                wms.append(O.FINAL_WATERMARK)
        for d in range(world):
            before = ctxs[d].last_present_watermark()
            for s in range(world):
                ctxs[d].watermarks.set(s, wms[s])
            after = ctxs[d].last_present_watermark()
            if after is not None and after != before:
                ops[d].handle_watermark(after, ctxs[d], outs[d])
    want_rows, want_sum = 0, 0
    for o in outs:
        for b in o.batches:
            want_rows += b.num_rows
            w = b["window"] if "window" in b.names() else None
            cols = [b["key"]] + ([w[:, 0], w[:, 1]] if w is not None else [b["window_start"], b["window_end"]]) + \
                [b["sum"], b["n"], b[O.TIMESTAMP]]
            want_sum = _i64(want_sum + _np_checksum(np, cols))
    ok = got == (want_rows, want_sum)
    return {"verified": ok, "rows_out": got[0], "expected_rows_out": want_rows,
            "against": f"oracle/arroyo_oracle.py session operator behind a simulated {world} x {world} shuffle",
            "checks": "sessions emitted and a wrapping checksum over every output column, summed over the owners",
            "size": f"{n_steps} steps of {srows} rows per GPU, {n_keys} keys per GPU, then end of data"}


def cpu_session(n_keys, srows, world, budget_s=20.0):
    """oracle/session_oracle.c, one single-threaded subtask per key partition (threads), on a bounded sample of the
    workload.  Returns (rows/s, threads, sample)."""
    from concurrent.futures import ThreadPoolExecutor

    import numpy as np

    from oracle import arroyo_oracle as O, c_oracle
    P = max(1, min(os.cpu_count() or 1, 64))
    warm, steps = 8, 4
    total_keys, total_rows = n_keys * world, srows * world
    while True:
        def work(q):
            rng = np.random.default_rng(100 + q)
            nk, nr = max(total_keys // P, 1), max(total_rows // P, 1)
            op = c_oracle.SessionAggregatingWindowFunc(_session_cfg(O))
            ctx, out = O.OperatorContext(1), O.Collector()
            sv = rng.integers(0, 10**6, nr, dtype=np.int64)
            offs = np.sort(rng.integers(0, S, nr, dtype=np.int64))
            t0 = None
            for p in range(warm + steps):
                if p == warm:
                    t0 = time.perf_counter()
                key = rng.integers(0, nk, nr, dtype=np.int64) * 7919
                op.process_batch(O.Batch({"key": key, "value": sv, O.TIMESTAMP: offs + (T0 + p * S)}), ctx, out)
                ctx.watermarks.set(0, T0 + p * S - S)
                op.handle_watermark(T0 + p * S - S, ctx, out)
                out.batches.clear()
            return (time.perf_counter() - t0) / steps

        t0 = time.perf_counter()
        with ThreadPoolExecutor(P) as pool:
            per_step = max(pool.map(work, range(P)))
        if time.perf_counter() - t0 <= budget_s or total_rows <= (1 << 18):
            return total_rows / per_step, P, (f"{steps} steps of {total_rows} rows over {total_keys} keys after {warm} warm-up "
                                              f"steps, {P} key-partitioned subtasks")
        total_keys //= 4
        total_rows //= 4


# ---------------------------------------------------------------------------------------------------------------
def run(args, B):
    import torch
    import torch.distributed as dist_mod

    from arroyo_b200 import ffi
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    all_cpus = os.sched_getaffinity(0)
    B.bind_to_gpu_numa_node(local)
    if ffi.load().arroyo_b200_device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: arroyo_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        dist_mod.init_process_group("nccl", device_id=device)
        dist = dist_mod
    torch.cuda.set_stream(torch.cuda.Stream(device=device))
    steps = args.steps
    sampler = B.ClockSampler(local) if rank == 0 else None
    if args.workload == "join":
        n_p, n_a, warm = 1 << args.join_persons_log2, 1 << args.join_auctions_log2, 3
        ms, rows_out, _, launches = _run_join(torch, dist, rank, world, local, device, n_p, n_a, warm, steps, 1,
                                              sampler=sampler)
        rows_step = n_p + n_a
        clocks = sampler.stop() if sampler is not None else None  # (before the verification pass sets its own edges up)
        verify = verify_join(torch, dist, rank, world, local, device)
        metric = "input rows/sec windowed hash-join (Nexmark q8 shape)"
        workload = (f"BASELINE configs[3]: q8-shaped 30-s tumbling person x auction join on person id = seller; every GPU's "
                    f"shard delivers {n_p} persons + {n_a} auctions per window; both inputs cross a key-hash shuffle")
        bytes_row = (24 * n_p + 32 * n_a) / rows_step
    else:
        n_keys, srows, warm = args.session_keys, 1 << args.session_rows_log2, 14
        ms, rows_out, _, launches = _run_session(torch, dist, rank, world, local, device, n_keys, srows, warm, steps, 1,
                                                 split=args.session_split, sampler=sampler)
        rows_step = srows
        clocks = sampler.stop() if sampler is not None else None
        verify = verify_session(torch, dist, rank, world, local, device)
        metric = "rows/sec session-window aggregate (5 s gap)"
        workload = (f"BASELINE configs[4]: session windows, gap 5 s, SUM + COUNT, {n_keys} keys per GPU; every GPU's shard "
                    f"delivers {srows} rows per second of event time; raw rows cross a key-hash shuffle")
        bytes_row = 24.0
    t = torch.tensor([ms, float(rows_out), float(launches)], dtype=torch.float64, device=device)
    if dist is not None:
        mx = t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(t)
        ms = float(mx[0].item())
        rows_out, launches = int(t[1].item()), int(t[2].item())
    if rank == 0:
        os.sched_setaffinity(0, all_cpus)
        cpu = None
        if not args.skip_cpu:
            if args.workload == "join":
                cpu = cpu_join(1 << args.join_persons_log2, 1 << args.join_auctions_log2, world)
            else:
                cpu = cpu_session(args.session_keys, 1 << args.session_rows_log2, world)
        value = world * steps * rows_step / (ms * 1e-3)
        peak, peak_kind = B.measured_peak()
        gbs = value * bytes_row / world / 1e9
        out = {"metric": metric, "value": value, "unit": "rows/s", "n_gpus": world, "steps": steps, "warmup": warm,
               "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
               "data": "synthetic",
               "config": {"workload": workload, "n_gpus": world,
                          "shuffle": ("csrc/exchange.cu round per input and step" if world > 1 else "one subtask: no repartition"),
                          "l2": "inputs larger than L2"},
               "rows_out_per_step": rows_out / max(steps, 1), "gpu_launches": launches,
               "roofline": {"bound": "hbm", "kernel": "whole operator step (not one kernel)", "achieved": round(gbs, 1),
                            "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": round(gbs / peak, 4), "traffic": None,
                            "note": f"{bytes_row:.1f} input bytes per row, per GPU, over the whole step"},
               "e2e": None, "clocks": clocks, "verify": verify, "verified": bool(verify and verify["verified"])}
        if cpu is not None:
            out["cpu_baseline"] = {"value": cpu[0], "unit": "rows/s", "cores": cpu[1], "kind": "port", "sample": cpu[2]}
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and not (verify and verify["verified"]):
        sys.exit("bench.py: GPU results differ from the oracle's -- see the verify block of the line above")
