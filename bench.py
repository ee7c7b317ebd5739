#!/usr/bin/env python
"""bench.py — rows/sec scanned and HBM GB/s of the group-by + histogram scan (BASELINE.json metric).

A "step" is one pass of the hot path (decode -> filter -> group-by -> aggregate ->
CombineResults) over one synthetic table.  The bench line is BASELINE.json configs[2] ("c3"):
1,000,000,000 rows, 3 ANDed int/str filters, group-by 2 columns, BasicHist on one column — the
configuration the metric is quoted on; it fits one B200 (32 GB encoded).  With N GPUs the same
1B rows are block-sharded over the ranks (strong scaling) and the per-group partials are merged
by one NCCL collective inside the timed step.  `--workload c2|c4|c5` selects another config
as the bench line; short runs of the others ride along in `extra` (c2: 100M rows per GPU, weak).

value     rows/s with the encoded blocks already resident in HBM when the timed region starts
          (inputs >> 126 MB of L2: no flush needed).
e2e       the same metric through the C ABI from pinned HOST buffers: every step re-stages all
          blocks (H2D inside the timed region), scans, and reads the result back.  Tables larger than
          the pinned arena go through it chunk by chunk; only the staging of each chunk, the
          scan and the result read-back are timed (chunks are regenerated between timed segments).
roofline  algorithmic bytes (8 B per int column, 4 B per str column referenced, SURVEY.md §8d)
          / scan-kernel time measured with CUDA events by the library.
parity    after the timed region rank 0 compares the (merged) result with an independent evaluation
          of the query on the generator's row values (blockgen.cpp sbg_eval: no encoding, no decode,
          no oracle): MatchedCount, every group's Count, hist Count, exact sum and bucket counter.
          A mismatch fails the run.
cpu_baseline  the CPU oracle (restatement of the reference's goroutine-per-block path; the Go
          reference cannot be built here) on a bounded sample, all host threads.

--dump-outputs DIR  writes what the last timed step of the bench line returned (MatchedCount, every group's
          key, Count, Samples and histogram fields, time buckets) as DIR/<name>.npy in float64, at most 64 MB.
          The tables are generated from fixed seeds, so two builds run with the same arguments can be compared
          array for array.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
import traceback

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "rows/sec scanned (group-by sum+hist scan)"
WORKLOADS = {
    "c2": "100M rows/GPU, group-by 1 str col (64 keys), sum+avg on 3 int cols",
    "c3": "1B rows, 3 ANDed int/str filters, group-by 2 cols, BasicHist on 1 col",
    "c4": "1B rows time series, 256 time buckets + per-bucket BasicHist",
    "c5": "high-cardinality group-by (1M distinct str keys), sum on 4 int cols",
}
SCALING = {"c2": "weak", "c3": "strong", "c4": "strong", "c5": "strong"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (default: the config's size)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--extra", default="auto", help="comma list of other configs to run briefly (auto: c2,c4,c5; none)")
    ap.add_argument("--selfcheck", action="store_true", help="multi-GPU: merged result of 4 small queries vs the oracle first")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step of the bench line as DIR/<name>.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's result (--impl ours)")
    return a


def total_rows_for(workload, world, rows_per_gpu, spec_rows):
    """Rows of the whole job: c2 is weak-scaled (100M rows per GPU), the 1B-row configs are strong-scaled."""
    if rows_per_gpu:
        return rows_per_gpu * world
    if workload == "c2":
        return 100_000_000 * world
    if workload == "c5":
        return min(spec_rows, 250_000_000 * world)  # 1M-key dictionaries intern ~65k strings per block on the host
    return spec_rows


def job_config(workload, world, total_rows, block_rows):
    """`config` of the JSON line — the same keys and values in both arms (`--impl reference` too)."""
    return {"workload": "%s: %s" % (workload, WORKLOADS.get(workload, "")), "total_rows": int(total_rows),
            "rows_per_gpu": int(total_rows // max(world, 1)), "block_rows": int(block_rows),
            "parallelism": "blocks sharded over %d GPU(s) + 1 NCCL merge" % world,
            "l2": "inputs larger than L2 (no flush)"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def seed_dicts(table, spec, F):
    """Identical key numbering on every rank (sg_table_dict_seed_*): the synthetic columns'
    value sets are known, so every rank seeds them in numeric order."""
    import numpy as np
    for c in spec.cols:
        if c.kind == F.SBG_STRKEY:
            strs = [(c.prefix + str(c.lo + v)).encode() for v in range(c.span)]
            offs = np.zeros(len(strs) + 1, np.uint32)
            offs[1:] = np.cumsum([len(s) for s in strs])
            blob = np.frombuffer(b"".join(strs), np.uint8)
            table.ctx.check(table.lib.sg_table_dict_seed_str(table.h, c.col_slot, blob.ctypes.data, offs.ctypes.data, len(strs)))
        elif c.kind == F.SBG_UNIFORM and c.span <= 5000:
            vals = np.arange(c.lo, c.lo + c.span, dtype=np.int64)
            table.ctx.check(table.lib.sg_table_dict_seed_int(table.h, c.col_slot, vals.ctypes.data, len(vals)))


def make_query(spec, synth):
    from tests.util import Q, Spec
    s = Spec(spec.key_table)
    s.IntInfo = dict(spec.IntInfo)
    kw = dict(synth.query_for(spec))
    # diagnostics only (scripts/gpu_ab.sh): SG_BENCH_OP=avg|hist, SG_BENCH_GROUPS=a,b override the config's query
    if os.environ.get("SG_BENCH_OP"):
        kw["op"] = os.environ["SG_BENCH_OP"]
    if os.environ.get("SG_BENCH_GROUPS") is not None:
        kw["groups"] = [g for g in os.environ["SG_BENCH_GROUPS"].split(",") if g]
    if spec.name == "c5":
        kw["limit"] = 100  # the reference CLI's default -limit (FLAGS.LIMIT): the top 100 of the 1M groups are materialised
    return Q(s, **kw)


DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much


def result_arrays(qs):
    """The fields of a materialised QuerySpec as float64 arrays.  Rows of `groups_*`: the Cumulative row, then
    the groups in the result's sorted order; rows of `time_*`: every (time bucket, group), buckets ascending and
    groups by key.  A key is the CRC-32 of its GroupByKey.  Counts and exact sums of the bench tables stay far
    below 2^53, so they convert exactly.  A group without a histogram holds NaN."""
    import zlib
    import numpy as np

    def padded(seqs):
        m = np.full((len(seqs), max((len(s) for s in seqs if s is not None), default=0)), np.nan)
        for i, s in enumerate(seqs):
            if s is not None:
                m[i, :len(s)] = s
        return m

    out = {"scalars": np.array([qs.MatchedCount, qs.NumGroups, qs.BrokenBlocks, qs.SkippedBlocks], np.float64)}
    tables = {"groups": [(None, r) for r in [qs.Cumulative] + qs.Sorted]}
    if qs.TimeResults:
        tables["time"] = [(tb, r) for tb, m in sorted(qs.TimeResults.items()) for _, r in sorted(m.items())]
        out["time_bucket"] = np.array([tb for tb, _ in tables["time"]], np.float64)
    for t, rows in tables.items():
        out[t + "_key_crc32"] = np.array([zlib.crc32(r.GroupByKey.encode()) for _, r in rows], np.float64)
        out[t + "_count"] = np.array([r.Count for _, r in rows], np.float64)
        out[t + "_samples"] = np.array([r.Samples for _, r in rows], np.float64)
        for a in qs.Aggregations:
            hs = [r.Hists.get(a.Name) for _, r in rows]
            for field, get in (("count", lambda h: h.TotalCount()), ("sum", lambda h: h.Sum()), ("min", lambda h: h.Min()),
                               ("max", lambda h: h.Max()), ("avg", lambda h: h.Mean()), ("stddev", lambda h: h.StdDev())):
                out["%s_%s_%s" % (t, a.Name, field)] = np.array([np.nan if h is None else get(h) for h in hs], np.float64)
            out["%s_%s_percentiles" % (t, a.Name)] = padded([None if h is None else h.GetPercentiles() for h in hs])
            out["%s_%s_buckets" % (t, a.Name)] = padded([None if h is None else h.Values for h in hs])
    return out


def sample_rows(arrays, limit=DUMP_BYTES):
    """Arrays larger than `limit` in all keep a fixed, seeded sample of the rows of each table; `<table>_rows`
    holds the indices kept.  Every row is at least 24 bytes, so the 8-byte index per row fits in the halved share."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total <= limit:
        return arrays
    rng = np.random.default_rng(0)
    for t in ("groups", "time"):
        names = [k for k in arrays if k.startswith(t + "_")]
        if names:
            n = len(arrays[names[0]])
            idx = np.sort(rng.choice(n, max(1, int(n * limit / (2 * total))), replace=False))
            for k in names:
                arrays[k] = arrays[k][idx]
            arrays[t + "_rows"] = idx.astype(np.float64)
    return arrays


def dump_outputs(path, table, qs):
    """--dump-outputs: materialise the result the last timed step kept (qs.result) and write its arrays."""
    import numpy as np
    try:
        qs.materialize = True
        table._fill(qs, qs.result)
    finally:
        table.lib.sg_result_free(qs.result)
        qs.result = None
    os.makedirs(path, exist_ok=True)
    for name, a in sample_rows(result_arrays(qs)).items():
        np.save(os.path.join(path, name + ".npy"), a)


def host_info():
    info = {"nproc": os.cpu_count()}
    try:
        info["sched_affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        info["numa_nodes"] = len(nodes)
    except Exception:
        pass
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    info["cpu"] = line.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    return info


class Env:
    """Process-wide state of one bench invocation: rank, context, the reusable pinned arena."""

    def __init__(self, args):
        import torch
        from sybil_b200 import engine as E
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        self.ctx = E.get_context(self.local)
        self.lib = self.ctx.lib
        if self.world > 1:
            uid = [self.ctx.comm_unique_id() if self.rank == 0 else None]
            self.dist.broadcast_object_list(uid, src=0)
            self.ctx.comm_init(uid[0], self.rank, self.world)
        self.arena, self.arena_bytes = None, 0

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def _reduce(self, x, op):
        if not self.dist:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX) if self.dist else x

    def sum_over_ranks(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM) if self.dist else x

    def pinned(self, nbytes):
        if nbytes > self.arena_bytes:
            if self.arena:
                self.lib.sg_pinned_free(self.ctx.h, self.arena)
            self.arena = self.lib.sg_pinned_alloc(self.ctx.h, nbytes)
            if not self.arena:
                raise RuntimeError("pinned arena: " + self.ctx.err())
            self.arena_bytes = nbytes
        return self.arena

    def close(self):
        if self.arena:
            self.lib.sg_pinned_free(self.ctx.h, self.arena)
            self.arena = None
        if self.dist:
            self.dist.destroy_process_group()


CHUNK_LIMIT = 12 << 30  # pinned arena the blocks are generated into and staged from


def run_workload(env, workload, rows_per_gpu, steps, warmup, do_e2e, e2e_steps, do_cpu, do_parity, dump_dir=None):
    """One config on this job's GPUs.  Returns the JSON line's fields (rank 0) or None (other ranks).
    dump_dir: rank 0 writes the result of the last timed step there (dump_outputs)."""
    from sybil_b200 import _ffi as F
    from sybil_b200 import engine as E
    from sybil_b200 import synth
    from sybil_b200.sharding import shard_range
    lib, ctx, world, rank = env.lib, env.ctx, env.world, env.rank

    base = synth.config(workload)
    total = total_rows_for(workload, world, rows_per_gpu, base.total_rows)
    spec = synth.config(workload, total_rows=total)
    nb_total = spec.num_blocks()
    first, nblocks = shard_range(nb_total, rank, world)
    bytes_per_row = synth.algorithmic_bytes_per_row(spec)

    # ---- inputs: generated on the host cores into pinned memory (untimed) ----------------
    per_block_bytes = spec.block_rows * (bytes_per_row + 8) + (1 << 21)
    chunk_blocks = max(1, min(nblocks, CHUNK_LIMIT // per_block_bytes))
    chunked = chunk_blocks < nblocks
    arena_bytes = chunk_blocks * per_block_bytes + (1 << 20)
    arena = env.pinned(arena_bytes)
    table = E.Table(workload, spec.key_table, ctx)
    table.IntInfo = dict(spec.IntInfo)
    if world > 1:
        seed_dicts(table, spec, F)
    gen_s = stage_s = 0.0
    my_rows = 0
    store = None

    def load(tbl, timed=None):
        """generate + stage every chunk of this rank's shard into `tbl`; timed(seconds) gets the staging time."""
        nonlocal store
        rows = 0
        g_s = s_s = 0.0
        for c0 in range(0, nblocks, chunk_blocks):
            if store is not None:
                store.close()
                store = None
            tg = time.perf_counter()
            nb = min(chunk_blocks, nblocks - c0)
            store = synth.generate(spec, first + c0, nb, arena_ptr=arena, arena_bytes=arena_bytes)
            ptrs, np_ = store.block_ptrs()
            for i in range(nb):
                rows += store.block(i).contents.num_records
            g_s += time.perf_counter() - tg
            env.torch.cuda.synchronize()
            ts = time.perf_counter()
            tbl.add_blocks(ptrs, np_)  # pinned host buffers -> HBM
            tbl.sync()
            s_s += time.perf_counter() - ts
        if timed is not None:
            timed(s_s)
        return rows, g_s, s_s

    my_rows, gen_s, stage_s = load(table)
    q = make_query(spec, synth)
    q.set_flags()

    prepared = {}

    def one_step(tbl, materialize=False, keep_result=False):
        """One query = one step.  The query is prepared once per table (QuerySpec -> sg_query_begin), as a host
        that repeats a dashboard query would; every step runs the scan, the merge and the result read-back."""
        qs = q.query_spec()
        qs.materialize = materialize  # the C library always builds the sorted result; the per-group
                                      # Python objects are only built for the checked step
        pq = prepared.get(id(tbl))
        if pq is None:
            ls = tbl.NewLoadSpec()
            for c in spec.cols:
                (ls.Int if c.col_type == F.SG_COL_INT else ls.Str)(c.name)
            pq = prepared[id(tbl)] = tbl.Prepare(ls, qs)
        pq.Run(qs, allreduce=world > 1, keep_result=keep_result)
        return qs

    # ---- value: resident inputs -----------------------------------------------------------
    for _ in range(warmup):
        qs = one_step(table)
    sampler = ClockSampler(env.local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    env.barrier()
    t0 = time.perf_counter()
    kernel_ms, launches = 0.0, 0
    keep_last = dump_dir is not None and rank == 0
    for i in range(steps):
        qs = one_step(table, keep_result=keep_last and i == steps - 1)
        kernel_ms += qs.stats.kernel_ms
        launches += qs.stats.kernel_launches
    env.barrier()
    elapsed = env.max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.finish() if sampler else None
    if keep_last:
        dump_outputs(dump_dir, table, qs)
    total_rows = env.sum_over_ranks(float(my_rows))
    ms_per_step = elapsed / steps * 1e3
    value = total_rows / (elapsed / steps)
    kernel_ms_avg = env.max_over_ranks(kernel_ms / steps)
    matched, ngroups = qs.MatchedCount, qs.NumGroups
    enc_bytes = int(lib.sg_table_encoded_bytes(table.h))

    # ---- parity: merged result vs the row-value evaluation (rank 0 checks; every rank runs the step) ----
    parity = None
    if do_parity:
        materialize = workload != "c5"  # 1M groups: checked through the bulk export below
        qs_chk = one_step(table, materialize=materialize)
        if rank == 0:
            t_chk = time.perf_counter()
            try:
                exp = synth.Expected(spec)
                if materialize:
                    n = exp.check(qs_chk)
                    what = "MatchedCount, group set, Count / hist Count / exact sum / every bucket counter of every group"
                else:
                    assert qs_chk.MatchedCount == exp.matched, ("MatchedCount", qs_chk.MatchedCount, exp.matched)
                    assert qs_chk.NumGroups == int((exp.count != 0).sum()), "number of groups"
                    n = 2
                    what = "MatchedCount and number of groups (1M groups: full comparison in tests/)"
                parity = {"checked": what, "values_compared": int(n), "ok": True, "rows": int(total_rows),
                          "against": "blockgen.cpp sbg_eval (query evaluated on the generator's row values)",
                          "seconds": round(time.perf_counter() - t_chk, 2)}
            except AssertionError as e:
                parity = {"ok": False, "error": repr(e)[:400]}

    # ---- e2e: host buffers -> H2D -> scan -> result, every step ---------------------------
    e2e = None
    if do_e2e:
        t2 = E.Table(workload + "_e2e", spec.key_table, ctx)
        t2.IntInfo = dict(spec.IntInfo)
        if world > 1:
            seed_dicts(t2, spec, F)
        e2e_ptrs = e2e_n = None
        if not chunked:
            e2e_ptrs, e2e_n = store.block_ptrs()

        def e2e_step():
            """returns (seconds inside timed segments, result, h2d bytes)"""
            ctx.check(lib.sg_table_clear(t2.h))
            env.torch.cuda.synchronize()
            seg = []
            if chunked:
                load(t2, timed=seg.append)  # every chunk: regenerate (untimed), stage (timed)
            else:
                ts = time.perf_counter()
                t2.add_blocks(e2e_ptrs, e2e_n)
                seg.append(time.perf_counter() - ts)
            ts = time.perf_counter()
            r = one_step(t2)  # waits for the copies, scans, merges, reads the result back
            seg.append(time.perf_counter() - ts)
            return sum(seg), r, lib.sg_table_h2d_bytes(t2.h)

        e2e_step()
        env.barrier()
        e_sum = 0.0
        for _ in range(e2e_steps):
            env.barrier()
            dt, r2, h2d = e2e_step()
            e_sum += env.max_over_ranks(dt)
        assert r2.MatchedCount == matched
        e2e = {"value": total_rows / (e_sum / e2e_steps), "unit": "rows/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(r2.stats.d2h_bytes), "steps": e2e_steps, "ms_per_step": e_sum / e2e_steps * 1e3,
               "timed": ("staging of each pinned chunk + scan + result (chunks regenerated between segments)" if chunked
                         else "re-stage all blocks + scan + result")}
        prepared.pop(id(t2)).Close()
        t2.close()

    out = None
    if rank == 0:
        # ---- roofline ---------------------------------------------------------------------------
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        achieved = my_rows * bytes_per_row / (kernel_ms_avg * 1e-3) / 1e9 if kernel_ms_avg > 0 else 0.0
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            ent = tj.get(workload)
            if isinstance(ent, dict):  # {"bytes_per_row": .., "source": ..}: scaled to this launch's rows
                traffic = ent.get("bytes_per_row", 0) * my_rows
                traffic_src = ent.get("source")
            elif ent is not None:
                traffic, traffic_src = ent, "profiles/traffic.json (ncu, r01)"
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "frac_of_nominal_8TBps": achieved / 8000.0, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peak_src, "kernel": "sg::scan_kernel", "kernel_ms_per_launch": kernel_ms_avg,
                    "algorithmic_bytes_per_row": bytes_per_row, "rows_per_launch": my_rows,
                    "encoded_bytes_resident": enc_bytes}
        cpu = None
        if do_cpu and world == 1:
            cpu = cpu_baseline(spec, store, q, store.num_blocks())
        out = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": SCALING.get(workload, "strong"), "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": job_config(workload, world, total_rows, spec.block_rows),
            "result": {"groups": int(ngroups), "matched_rows": int(matched), "blocks_per_gpu": int(nblocks)},
            "hbm_gbps": achieved * world, "roofline": roofline, "parity": parity, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": int(launches), "clocks": clocks,
            "setup": {"generate_s": round(gen_s, 2), "stage_s": round(stage_s, 2)},
        }
    for pq in prepared.values():
        pq.Close()
    table.close()
    if store is not None:
        store.close()
    return out


def selfcheck(env):
    """tests/multi_gpu_check.py inside the bench: four small queries, seeded and per-rank dictionaries,
    merged over this job's GPUs and compared with the oracle over all blocks (rank 0)."""
    from sybil_b200.sharding import shard_range
    from tests.multi_gpu_check import run_mode
    from tests.util import Q, random_spec
    spec = random_spec(123, nrows=40000, block_rows=2500)
    queries = [
        Q(spec, groups=["host"], aggs=["age", "lat", "big"], op="avg"),
        Q(spec, int_filters=[("age", "gt", 12)], str_filters=[("state", "neq", "s3")], groups=["host", "age"], aggs=["lat"], op="hist"),
        Q(spec, groups=["state"], aggs=["big"], op="hist", loghist=True),
        Q(spec, groups=["host"], aggs=["lat"], op="hist", time_col="time", time_bucket=600),
    ]
    first, count = shard_range(len(spec.blocks), env.rank, env.world)
    ok = True
    for seeded in (True, False):
        ok &= run_mode(env.ctx, spec, queries, first, count, env.rank, env.world, seeded, quiet=True)
    return {"queries": len(queries), "dictionary_modes": ["seeded", "per-rank"], "ok": bool(ok),
            "against": "oracle over all blocks (tests/multi_gpu_check.py)"}


def run_ours(args):
    env = Env(args)
    sc = None
    if env.world > 1 or args.selfcheck:
        try:
            sc = selfcheck(env)
        except Exception as e:  # noqa: BLE001
            sc = {"ok": False, "error": repr(e)[:300]}
    line = run_workload(env, args.workload, args.rows, args.steps, args.warmup, not args.no_e2e, args.e2e_steps,
                        not args.no_cpu, not args.no_parity, args.dump_outputs)
    extras = []
    names = [] if args.extra == "none" else (["c2", "c4", "c5"] if args.extra == "auto" else args.extra.split(","))
    if args.rows and args.extra == "auto":
        names = []  # an experiment at a custom size: just that line
    for w in names:
        if w == args.workload or w not in WORKLOADS:
            continue
        try:
            x = run_workload(env, w, 0, max(3, min(args.steps, 10)), 3, False, 0, False, not args.no_parity)
        except Exception as e:  # noqa: BLE001
            x = {"config": {"workload": w}, "error": repr(e)[:300], "trace": traceback.format_exc()[-600:]}
        if x is not None:
            keep = ("value", "unit", "ms_per_step", "scaling", "config", "result", "hbm_gbps", "roofline", "parity", "gpu_launches",
                    "error", "trace", "steps", "warmup")
            extras.append({k: x[k] for k in keep if k in x})
    if env.rank == 0:
        line["extra"] = extras
        line["multi_gpu_selfcheck"] = sc
        line["host"] = host_info()
        bad = [p for p in [line.get("parity")] + [x.get("parity") for x in extras] if p is not None and not p.get("ok")]
        if sc is not None and not sc.get("ok"):
            bad.append(sc)
        print(json.dumps(line))
        sys.stdout.flush()
        env.close()
        if bad:
            print("PARITY FAILURE: %r" % (bad,), file=sys.stderr)
            sys.exit(1)
    else:
        env.close()


def cpu_baseline(spec, store, q, nblocks, target_s=15.0):
    """The oracle (CPU restatement of the reference path) on a bounded sample of the same blocks."""
    from oracle.oracle_ffi import OracleTable, lib as olib
    threads = olib().orc_hardware_threads()
    d, keep = q.desc()
    probe = min(nblocks, max(threads, 8))
    ot = OracleTable(spec.key_table)
    for i in range(probe):
        ot.add_block(store.block(i))
    r = ot.query(d, q.aggs, nthreads=threads, details=False)
    rows_probe = sum(store.block(i).contents.num_records for i in range(probe))
    rate = rows_probe / max(r.seconds, 1e-6)
    want = int(min(nblocks, max(probe, rate * target_s / spec.block_rows)))
    for i in range(probe, want):
        ot.add_block(store.block(i))
    r = ot.query(d, q.aggs, nthreads=threads, details=False)
    rows = sum(store.block(i).contents.num_records for i in range(want))
    ot.close()
    return {"value": rows / r.seconds, "unit": "rows/s", "cores": threads, "kind": "port", "threads_used": threads,
            "host": host_info(),
            "sample": "%d blocks (%d rows) of the same table, %.1f s" % (want, rows, r.seconds)}


def run_reference(args):
    """--impl reference: the reference's CPU path (its C++ restatement: no Go toolchain in this
    image, see DESIGN.md) on the host cores, same workload/metric, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sybil_b200 import synth
    from oracle.oracle_ffi import OracleTable, lib as olib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    base = synth.config(args.workload)
    total = total_rows_for(args.workload, world, args.rows, base.total_rows)
    spec = synth.config(args.workload, total_rows=total)
    threads = olib().orc_hardware_threads()
    q = make_query(spec, synth)
    q.set_flags()
    d, keep = q.desc()
    # calibrate a sample that keeps warmup+steps within a few minutes
    probe = min(spec.num_blocks(), max(threads, 8))
    store = synth.generate(spec, 0, probe)
    ot = OracleTable(spec.key_table)
    for i in range(probe):
        ot.add_block(store.block(i))
    r = ot.query(d, q.aggs, nthreads=threads, details=False)
    rate = probe * spec.block_rows / max(r.seconds, 1e-6)
    budget_s = 120.0 / max(args.steps + args.warmup, 1)
    want = int(min(spec.num_blocks(), max(probe, rate * min(budget_s, 10.0) / spec.block_rows)))
    if want > probe:
        store.close()
        ot.close()
        store = synth.generate(spec, 0, want)
        ot = OracleTable(spec.key_table)
        for i in range(want):
            ot.add_block(store.block(i))
    rows = sum(store.block(i).contents.num_records for i in range(want))
    for _ in range(args.warmup):
        ot.query(d, q.aggs, nthreads=threads, details=False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ot.query(d, q.aggs, nthreads=threads, details=False)
    el = time.perf_counter() - t0
    value = rows * args.steps / el
    sample = "first %d blocks (%d rows) of the table per step" % (want, rows)
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3,
           "higher_is_better": True, "scaling": SCALING.get(args.workload, "strong"), "vs_baseline": None, "dtype": "int64",
           "data": "synthetic", "config": job_config(args.workload, world, total, spec.block_rows),
           "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample,
                            "threads_used": threads, "host": host_info()},
           "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


if __name__ == "__main__":
    a = parse()
    import __graft_entry__
    __graft_entry__.build()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
