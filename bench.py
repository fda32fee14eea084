#!/usr/bin/env python
"""bench.py -- the hot-path benchmark (contract in the task brief, metric from BASELINE.json).

Headline (N=1): BASELINE.json configs[1] -- 100 M-row, 8-column synthetic table, 2 predicates ->
GROUP BY (1e5 keys) SUM/AVG/COUNT, in Mrows/s. The same JSON line carries a `bm25` object for
configs[2] -- 10 M-doc synthetic Zipf corpus, batch of two-term disjunctive BM25 top-1000 queries, in
Mdocs/s (postings scanned per second) -- because BASELINE.json's metric names both.

  value     whole step with inputs resident in HBM, device-timed on the library's stream
  e2e       the same metric through the public host API with HOST buffers (H2D of the step's inputs
            from pinned memory + D2H of the results inside the timed region)
  roofline  dominant kernel: algorithmic bytes per launch / CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline / --impl reference
            the CPU oracle (oracle/, a restatement of the reference's operators: the reference itself
            needs clang-21 + DuckDB + Abseil and cannot be built here) on the box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

K, A, B, V, W_ = 10, 11, 12, 13, 14          # field ids of the referenced columns k, a, b, v, w
COLS = {K: (10, 0, np.int64), A: (11, 1, np.int64), B: (12, 2, np.float64), V: (13, 3, np.int64), W_: (14, 4, np.float64)}
UNREFERENCED = {15: (15, 5), 16: (16, 5), 17: (17, 5)}  # c5..c7: part of the 8-column table, never read
N_TERMS = 256
TOPK = 1000


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and clock-event reasons sampled while a timed region runs. The nvidia-smi clocks line of the profiling
    recipe needs ~100 ms per sample, longer than a short timed region (10 steps of 1 ms), so the same counters are also read
    straight from NVML by a thread every 2 ms; nvidia-smi rows are merged in when any arrive."""

    def __init__(self, device, enabled=True):
        self.device = device
        self.enabled = enabled    # multi-GPU runs sample on rank 0 only: eight pollers on one driver are eight too many
        self.proc = None
        self.path = None
        self.rows = []          # (sm_mhz, max_mhz, reasons bitmask) from NVML
        self._stop = threading.Event()
        self._thr = None
        self._nv = None

    def _nvml_loop(self):
        nv, h = self._nv
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        while not self._stop.is_set():
            try:
                self.rows.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), mx, int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))))
            except Exception:
                break
            self._stop.wait(0.004)

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            import pynvml as nv
            nv.nvmlInit()
            self._nv = (nv, nv.nvmlDeviceGetHandleByIndex(int(self.device)))
            self._thr = threading.Thread(target=self._nvml_loop, daemon=True)
            self._thr.start()
        except Exception:
            self._nv = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device),
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        sm, reasons = [], set()
        try:
            rows = [l.strip().split(", ") for l in open(self.path) if l.strip()]
            os.unlink(self.path)
            sm += [float(r[0]) for r in rows]
            if rows:
                out["sm_max_mhz"] = float(rows[0][1])
            for i, nme in enumerate(names):
                if any(r[3 + i].strip().lower().startswith("active") for r in rows):
                    reasons.add(nme)
        except Exception:
            pass
        if self.rows and self._nv is not None:
            nv = self._nv[0]
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            sm += [r[0] for r in self.rows]
            if out["sm_max_mhz"] is None and self.rows[0][1] is not None:
                out["sm_max_mhz"] = float(self.rows[0][1])
            for nme, bit in bits.items():
                if any(r[2] & bit for r in self.rows):
                    reasons.add(nme)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["samples"] = len(sm)
            out["reasons"] = [n for n in names if n in reasons]
        return out


def merge_clocks(a, b):
    if not a.get("samples"):
        return b
    if not b.get("samples"):
        return a
    return {"sm_mhz": float(np.median([a["sm_mhz"], b["sm_mhz"]])), "sm_max_mhz": a["sm_max_mhz"],
            "reasons": sorted(set(a["reasons"]) | set(b["reasons"])), "samples": a["samples"] + b["samples"]}


def ncu_traffic(kernel, units):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed `ncu --set full`
    capture of this command (profiles/traffic.json names the capture); null when the workload size differs
    from the captured one or no capture is recorded."""
    try:
        t = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")))[kernel]
        return t["dram_bytes"] if int(t["units"]) == int(units) else None
    except Exception:
        return None


_M64 = (1 << 64) - 1


def synth_hash(stream, index):
    """splitmix64 finaliser over seed ^ (stream << 48) ^ index (SURVEY §8d) -- the generator both the product and the
    oracle use; restated here so that the query list depends on neither library."""
    z = ((0x5EDB2026 ^ ((stream << 48) & _M64) ^ index) + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, groups, keys, nq):
    """Writes what the timed paths returned in their last step as float32 / float64 .npy files, so that two builds can be
    compared output for output: the GROUP BY rows (the 128-bit SUM(v) rounded to float64), and each query's top-k decoded
    from its sortable keys in hit order (score desc, doc asc; doc -1 marks an empty slot). If the top-k arrays would not
    fit in DUMP_BYTES, a fixed seeded sample of the queries is written, with their indices in bm25_query."""
    import serenedb_b200 as sdb
    out = {}
    if groups is not None:
        out["groupby_key"] = groups["key"].astype(np.float64)
        out["groupby_count"] = groups["count"].astype(np.float64)
        out["groupby_sum_v"] = np.array([float(s) for s in sdb.sum_i128(groups)], np.float64)
        out["groupby_sum_w"] = groups["sum_f64"].astype(np.float64)
        out["groupby_count_w"] = groups["cnt_f64"].astype(np.float64)
    if keys is not None:
        k = keys.view(np.uint64).reshape(nq, -1)
        room = DUMP_BYTES - sum(a.nbytes for a in out.values()) - (1 << 16)   # headroom for the .npy headers
        take = min(nq, room // (k.shape[1] * 12 + 8))
        q = np.arange(nq) if take == nq else np.sort(np.random.default_rng(0).choice(nq, take, replace=False))
        k = np.sort(k[q], axis=1)[:, ::-1]
        doc = (~k & np.uint64(0xFFFFFFFF)).astype(np.float64)
        doc[k == 0] = -1
        out["bm25_query"] = q.astype(np.float64)
        out["bm25_score"] = (k >> np.uint64(32)).astype(np.uint32).view(np.float32)
        out["bm25_doc"] = doc
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def make_queries(nq, n_terms=N_TERMS, stream=7):
    """Two-term disjunctions, pairs drawn from the synthetic terms (SURVEY §8d); query 0 is the named
    case p = (0.10, 0.01) => terms 5 and 59."""
    qs = [[5, 59]]
    i = 0
    while len(qs) < nq:
        a = synth_hash(stream, 2 * i) % n_terms
        b = synth_hash(stream, 2 * i + 1) % n_terms
        i += 1
        if a != b:
            qs.append([int(a), int(b)])
    return qs


# --------------------------------------------------------------------------------------------
# CPU legs (the oracle; the only place bench.py touches oracle/)
# --------------------------------------------------------------------------------------------
def cpu_groupby(host_cols, rows, threads, reps):
    import orc
    seg = orc.Segment(rows, has_wand=False)
    for f, arr in host_cols.items():
        seg.add_column(f, arr[:rows])
    preds = [orc.make_pred(A, "LT", 500000), orc.make_pred(B, "GE", 0.25, is_float=True)]
    times = []
    out = None
    for _ in range(reps):
        t = time.perf_counter()
        out = orc.filter_groupby([seg], preds, K, V, W_, cap=100001, threads=threads)
        times.append(time.perf_counter() - t)
    return out, times


def cpu_bm25_setup(n_docs, threads):
    import orc
    orc.use_simdcomp_ref(True)  # decode 128-value blocks with the reference's own SSE simdcomp when oracle/_ref exists
    seg, dc, sum_dl = orc.synth_segment_mt(n_docs, 0, N_TERMS, doc0=0, threads=threads)
    return seg, dc, sum_dl


def cpu_bm25(seg, dc, sum_dl, n_docs, queries, threads, mode=2):
    import orc
    qt = []
    for q in queries:
        ts = []
        for t in q:
            st = orc.bm25_stats(n_docs, sum_dl, int(dc[t]))
            x = orc.BM25Term()
            x.idf, x.norm_const, x.norm_length, x.boost, x.term = st.idf, st.norm_const, st.norm_length, 1.0, t
            ts.append(x)
        qt.append(ts)
    t = time.perf_counter()
    hits, n_out, total, scored = orc.bm25_topk_batch([seg], "OR", qt, TOPK, mode=mode, threads=threads)
    return time.perf_counter() - t, hits, n_out, scored


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# --------------------------------------------------------------------------------------------
def run_reference(args, rank):
    """--impl reference: the reference path's CPU implementation (oracle port) on all host cores."""
    if rank != 0:
        return
    cores = host_cores()
    threads = min(cores, args.cpu_threads or cores)
    rows = args.cpu_rows
    cols = {f: None for f in COLS}
    import orc
    for f, (stream, kind, _) in COLS.items():
        cols[f] = orc.synth_column(stream, kind, 0, rows)
    # warm-up doubles as a thread-count probe: the port may peak below the full hyper-thread count
    probe = {thr: min(cpu_groupby(cols, rows, thr, 2)[1]) for thr in sorted({threads, max(1, threads // 2), max(1, threads // 4)})}
    threads = min(probe, key=probe.get)
    _, times = cpu_groupby(cols, rows, threads, max(1, args.warmup - 2) + args.steps)
    t = times[max(1, args.warmup - 2):]
    ms = 1e3 * float(np.mean(t))
    val = rows / np.mean(t) / 1e6
    line = {"impl": "reference", "metric": "filter->GROUP BY throughput (BASELINE.json configs[1]; bm25 object = configs[2])", "value": round(val, 2),
            "unit": "Mrows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
            "config": {"workload": "groupby: %d rows/GPU x 8 int64/float64 columns (5 referenced, 40 B/row), a<500000 AND b>=0.25 -> "
                                   "GROUP BY k (1e5 keys) SUM(v), AVG(w), COUNT(*)" % args.rows,
                       "rows_per_gpu": args.rows, "sample_rows": rows},
            "cpu_baseline": {"value": round(val, 2), "unit": "Mrows/s", "cores": threads, "kind": "port",
                             "sample": "%d-row prefix of the same synthetic table per step (oracle restatement; the reference "
                                       "binary needs clang-21+DuckDB+Abseil and cannot be built here)" % rows},
            "e2e": {"value": round(val, 2), "unit": "Mrows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not args.skip_bm25:
        seg, dc, sum_dl = cpu_bm25_setup(args.docs, threads)
        qs = make_queries(args.queries)[: args.cpu_queries]
        postings = sum(int(dc[a]) + int(dc[b]) for a, b in qs)
        ts = []
        for i in range(args.warmup + args.steps):
            dt, _, _, _ = cpu_bm25(seg, dc, sum_dl, args.docs, qs, threads)
            ts.append(dt)
        t = ts[args.warmup:]
        line["bm25"] = {"metric": "BM25 top-1000, 2-term OR batch: postings scanned per second (BASELINE.json configs[2])", "value": round(postings / np.mean(t) / 1e6, 2),
                        "unit": "Mdocs/s", "ms_per_step": round(1e3 * float(np.mean(t)), 3),
                        "cpu_baseline": {"value": round(postings / np.mean(t) / 1e6, 2), "unit": "Mdocs/s", "cores": threads, "kind": "port",
                                         "sample": "%d of the %d two-term OR queries per step, block-max pruned oracle, simdcomp unpack from oracle/_ref"
                                                   % (len(qs), args.queries)}}
    emit_line(line)


_JSON_FD = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout. Libraries (NCCL prints its version banner there) get stderr:
    fd 1 is pointed at fd 2 for the whole run and the line is written to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline GROUP BY and BM25 legs and of their e2e legs; the secondary probes "
                         "(BM25 pruning-off roofline, HBM-resident index, zonemap, configs[0], configs[3]) keep fixed counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="table rows per GPU")
    ap.add_argument("--docs", type=int, default=10_000_000, help="corpus docs per GPU")
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--skip-bm25", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="kernel probes only (no host round trip)")
    ap.add_argument("--skip-extra", action="store_true", help="skip BASELINE configs[0] and configs[3]")
    ap.add_argument("--cpu-rows", type=int, default=100_000_000)
    ap.add_argument("--cpu-queries", type=int, default=256)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (float32/float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # BASELINE configs[4]: 1 B rows / 100 M docs sharded 8 ways = 125 M rows and 12.5 M docs per GPU (weak scaling:
        # the per-GPU shard is the same at every N > 1); N = 1 runs configs[1] / configs[2] at their own sizes.
        if args.rows == 100_000_000:
            args.rows = 125_000_000
        if args.docs == 10_000_000:
            args.docs = 12_500_000
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.impl == "reference":
        args.cpu_rows = min(args.cpu_rows, args.rows)
        run_reference(args, rank)
        return

    import torch
    import serenedb_b200 as sdb
    from serenedb_b200 import dist as sd

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    ctx = sdb.Context(local)
    hbm_peak, peak_src = peaks()
    merge_via = "none"
    if dist is not None:
        # The collectives run inside libsdbg.so (sdbg_dist_*: NCCL on the context's stream, no host sync between the
        # partial kernel, the all-reduce and the next kernel); torch.distributed only carries the 128-byte NCCL id.
        try:
            idt = torch.zeros(128, dtype=torch.uint8, device=dev)
            if rank == 0:
                idt.copy_(torch.frombuffer(bytearray(sdb.Context.dist_unique_id()), dtype=torch.uint8))
            dist.broadcast(idt, 0)
            ctx.dist_init(bytes(idt.cpu().numpy().tobytes()), rank, world)
            merge_via = "sdbg_dist (NCCL from the C ABI)"
        except Exception as e:                      # pragma: no cover -- keeps the multi-GPU line alive if NCCL cannot be dlopened
            sys.stderr.write("sdbg_dist_init failed (%s): falling back to torch.distributed collectives\n" % e)
            merge_via = "torch.distributed"

    def barrier():
        torch.cuda.synchronize()
        ctx.sync()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ------------------------------------------------------------------ table shard in HBM
    rows = args.rows
    row0 = rank * rows
    seg = sdb.Segment(ctx, rows)
    for f, (stream, kind, _) in COLS.items():
        seg.synth_column(f, stream, kind, row0, rows)
    for f, (stream, kind) in UNREFERENCED.items():
        seg.synth_column(f, stream, kind, row0, rows)
    ctx.sync()
    scan = sdb.IResearchScan([seg])
    preds = [sdb.pred(A, "LT", 500000), sdb.pred(B, "GE", 0.25)]
    key_min, span = 0, 100000
    d_i64 = torch.zeros(4 * span, dtype=torch.int64, device=dev)
    d_f64 = torch.zeros(span, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()

    w_bound = 1000.0 * rows * world      # |SUM(w)| <= max|w| * total rows: fixes the fixed-point unit of the merged double sums

    def groupby_step():
        # device-resident step: columns in HBM -> dense partial aggregates in HBM (merged across ranks)
        scan.groupby_partial(preds, K, key_min, span, V, W_, d_i64.data_ptr(), d_f64.data_ptr())
        if dist is not None:
            if merge_via.startswith("sdbg_dist"):   # ONE all-reduce (counts + SUM(int) limbs + SUM(double) as fixed point), same stream
                ctx.dist_groupby_merge(d_i64.data_ptr(), d_f64.data_ptr(), span, w_bound)
            else:
                ctx.sync()
                sd.merge_groupby_partials(dist, d_i64, d_f64)
                torch.cuda.synchronize()

    def groupby_result():
        return scan.groupby_finalize(key_min, span, d_i64.data_ptr(), d_f64.data_ptr(), span)

    for _ in range(args.warmup):
        groupby_step()
    barrier()
    ctx.profile(True)
    launches0 = ctx.launches
    with ClockSampler(local, rank == 0) as cs1:
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            groupby_step()
        ms_total = ctx.timer_stop()
        res = groupby_result()
        barrier()
    gb_ms = max_over_ranks(ms_total) / args.steps
    k_ms, k_n = ctx.profile_read("groupby")
    ctx.profile(False)
    gb_launches = ctx.launches - launches0
    clocks = cs1.summary()
    gb_value = world * rows / (gb_ms * 1e-3) / 1e6
    gb_kernel_ms = k_ms / max(k_n, 1)
    gb_alg_bytes = rows * 40 + span * 32          # 5 referenced 8-byte columns + the 3.2 MB group table
    gb_ach = gb_alg_bytes / (gb_kernel_ms * 1e-3) / 1e9
    n_groups = len(res)
    n_pass = int(res["count"].sum())

    gb_e2e, e_ms, e_steps, h2d, d2h, host = None, None, 0, rows * 40, 0, {}
    if not args.skip_e2e:
        # ------------------------------------------------------------------ e2e: host columns -> host groups
        host = {}
        for f, (_, _, dt) in COLS.items():
            h = torch.empty(rows, dtype=torch.int64 if dt == np.int64 else torch.float64, pin_memory=True)
            seg.column_to_host(f, h.data_ptr(), rows)
            host[f] = h
        torch.cuda.synchronize()
        eseg = sdb.Segment(ctx, rows)
        escan = sdb.IResearchScan([eseg])
        d2h = None
        # The integer columns travel in their storage encoding (frame-of-reference bit-packing in 2048-row groups, the
        # algorithm of the reference's DuckDB `bitpacking` column codec): packed once on the host, outside the timed
        # region -- that is how they sit in the `.col` file / page cache -- and unpacked on the GPU after the copy. The
        # float64 columns are random mantissas and travel raw. `e2e_raw` repeats the measurement with every column raw.
        packed = {}
        for f, (_, _, dt) in COLS.items():
            if dt == np.int64:
                wbuf = torch.empty(rows + 1, dtype=torch.int64, pin_memory=True)
                hd, wd, _ = sdb.pack_for(host[f].numpy(), out_words=wbuf.numpy().view(np.uint64))
                hbuf = torch.empty(len(hd) * 2, dtype=torch.int64, pin_memory=True)
                hview = hbuf.numpy().view(sdb.engine.FOR_BLOCK_DTYPE)
                hview[:] = hd
                packed[f] = (hview, wd, rows, wbuf, hbuf)
        h2d_packed = sum(p[0].nbytes + p[1].nbytes for p in packed.values()) + sum(rows * 8 for f in COLS if f not in packed)
        h2d_raw = rows * 40

        def e2e_step(use_packed=True):
            for f, (_, _, dt) in COLS.items():
                if use_packed and f in packed:
                    eseg.stage_column_for(f, packed[f][:3])
                else:
                    eseg.stage_column(f, (host[f].data_ptr(), dt, rows))
            if dist is None:
                return escan.groupby(preds, K, sum_int_field=V, avg_f64_field=W_, cap=span, n_groups_hint=span)
            escan.groupby_partial(preds, K, key_min, span, V, W_, d_i64.data_ptr(), d_f64.data_ptr())
            if merge_via.startswith("sdbg_dist"):
                ctx.dist_groupby_merge(d_i64.data_ptr(), d_f64.data_ptr(), span, w_bound)
            else:
                ctx.sync()
                sd.merge_groupby_partials(dist, d_i64, d_f64)
                torch.cuda.synchronize()
            return escan.groupby_finalize(key_min, span, d_i64.data_ptr(), d_f64.data_ptr(), span)

        e_steps = args.steps
        e_raw_ms = None
        for use_packed in (False, True):
            eres = e2e_step(use_packed)
            eres = e2e_step(use_packed)
            barrier()
            ctx.timer_start()
            for _ in range(e_steps):
                eres = e2e_step(use_packed)
            t_ms = max_over_ranks(ctx.timer_stop()) / e_steps
            barrier()
            assert np.array_equal(eres["count"], res["count"]) and np.array_equal(eres["sum_lo"], res["sum_lo"])
            if use_packed:
                e_ms = t_ms
            else:
                e_raw_ms = t_ms
        h2d = h2d_packed
        d2h = int(len(eres)) * 48 + 16
        assert np.array_equal(eres["count"], res["count"]) and np.array_equal(eres["sum_lo"], res["sum_lo"])
        gb_e2e = world * rows / (e_ms * 1e-3) / 1e6
        eseg.close()

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1)
    cpu_gb = None
    cores = host_cores()
    threads = min(cores, args.cpu_threads or cores)
    if rank == 0 and world == 1 and not args.skip_cpu and not args.skip_e2e:
        crow = min(args.cpu_rows, rows)
        cols = {f: host[f].numpy() for f in COLS}
        cres, ctimes = cpu_groupby(cols, crow, threads, 3)
        best, best_thr = min(ctimes), threads
        for thr2 in (max(1, threads // 2), max(1, threads // 4)):   # hyper-threads / NUMA: the port may peak below the full thread count
            c2, t2 = cpu_groupby(cols, crow, thr2, 2)
            if min(t2) < best:
                best, best_thr = min(t2), thr2
        cpu_gb = {"value": round(crow / best / 1e6, 2), "unit": "Mrows/s", "cores": best_thr, "kind": "port",
                  "sample": "%d rows of the same table, best of 3 (oracle restatement of the scan+DuckDB aggregate)" % crow}
        if crow == rows:  # the CPU leg doubles as a full-size parity check of this very run
            assert np.array_equal(cres["key"], res["key"]) and np.array_equal(cres["count"], res["count"])
            assert np.array_equal(cres["sum_lo"], res["sum_lo"]) and np.array_equal(cres["sum_hi"], res["sum_hi"])
            assert np.allclose(cres["sum_f64"] / cres["cnt_f64"], res["sum_f64"] / res["cnt_f64"], rtol=1e-5)
    del host

    line = {
        "metric": "filter->GROUP BY throughput (BASELINE.json configs[1]; bm25 object = configs[2])",
        "value": round(gb_value, 1), "unit": "Mrows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(gb_ms, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64+f64", "data": "synthetic",
        "config": {"workload": "groupby: %d rows/GPU x 8 int64/float64 columns (5 referenced, 40 B/row), a<500000 AND b>=0.25 -> "
                               "GROUP BY k (1e5 keys) SUM(v), AVG(w), COUNT(*)" % rows,
                   "rows_per_gpu": rows, "groups": n_groups, "rows_passing": n_pass, "parallelism": "row-range shards x%d" % world,
                   "l2": "inputs (%.1f GB/GPU) larger than L2; no flush needed" % (rows * 40 / 1e9),
                   "merge": "none" if world == 1 else ("1 NCCL all-reduce per step (counts | SUM(int) limbs | SUM(double) as 120-bit fixed point in one int64 buffer), "
                                                         "enqueued by libsdbg.so on the kernel's stream" if merge_via.startswith("sdbg_dist")
                                                         else "2 torch.distributed all-reduces per step (fallback)")},
        "clocks": clocks,
        "e2e": None if gb_e2e is None else {"value": round(gb_e2e, 1), "unit": "Mrows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                               "ms_per_step": round(e_ms, 3), "steps": e_steps,
                                               "h2d_encoding": "int64 columns k, a, v frame-of-reference bit-packed in 2048-row groups (17 / 20 / 11 bits per value; packed on the host "
                                                               "outside the timed region, unpacked on the GPU inside it), float64 columns b, w raw",
                                               "e2e_raw": {"value": round(world * rows / (e_raw_ms * 1e-3) / 1e6, 1), "unit": "Mrows/s", "h2d_bytes_per_step": h2d_raw,
                                                           "ms_per_step": round(e_raw_ms, 3), "note": "every column copied as raw 8-byte values"}},
        "gpu_launches": int(gb_launches),
        "roofline": {"bound": "hbm", "achieved": round(gb_ach, 1), "peak": hbm_peak, "unit": "GB/s",
                     "frac": round(gb_ach / hbm_peak, 4), "traffic": ncu_traffic("filter_groupby_tma_kernel", rows), "kernel": "filter_groupby_tma_kernel",
                     "kernel_ms": round(gb_kernel_ms, 4), "algorithmic_bytes": gb_alg_bytes, "peak_source": peak_src},
    }
    if cpu_gb:
        line["cpu_baseline"] = cpu_gb

    oseg = odc = osdl = None
    bm25_keys, nq = None, 0
    # ------------------------------------------------------------------ BM25 (configs[2])
    if not args.skip_bm25:
        n_docs = args.docs
        cseg = sdb.Segment(ctx, n_docs)
        dc, sum_dl = cseg.synth_corpus(rank * n_docs, 0, N_TERMS, threads=min(cores, 64))
        dct = torch.tensor(dc.astype(np.int64), device=dev)
        sdl = torch.tensor([sum_dl], dtype=torch.int64, device=dev)
        ndf = torch.tensor([n_docs], dtype=torch.int64, device=dev)
        # corpus-wide statistics: summed once at index-build time (collectors.cpp:36-52), not per query
        sd.global_term_stats(dist, dct, sdl, ndf)
        reader = sdb.IndexReader([cseg], int(ndf.item()), int(sdl.item()), dct.cpu().numpy())
        scorer = sdb.BM25(1.2, 0.75)
        queries = make_queries(args.queries)
        batch = sdb.PreparedBatch(reader, queries, sdb.OR, scorer, TOPK)
        nq = len(queries)
        postings = int(sum(int(dc[a]) + int(dc[b]) for a, b in queries))
        tb = cseg.term_bytes(N_TERMS)
        list_bytes = int(sum(int(tb[a]) + int(tb[b]) + int(dc[a]) + int(dc[b]) for a, b in queries))
        alg_bytes = list_bytes + nq * TOPK * 12
        keys = torch.zeros(nq * TOPK, dtype=torch.int64, device=dev)
        keys_all = torch.zeros(world * nq * TOPK, dtype=torch.int64, device=dev) if dist is not None else None
        via_c = dist is not None and merge_via.startswith("sdbg_dist")

        def bm25_step(to_host=False):
            if via_c:     # scan -> ONE all-gather of the k best keys per query -> local selection, all on the library's stream
                return batch.run_dist(to_host=to_host)
            batch.run_device(rank, keys.data_ptr())
            if dist is not None:
                sd.gather_topk_keys(dist, keys, keys_all)
                torch.cuda.synchronize()
                return sdb.merge_gathered(ctx, keys_all.data_ptr(), world, nq, TOPK, to_host=to_host)
            return None

        def timed_bm25(step, steps, what):
            """-> (ms per step, top-k kernel ms per step, merge kernel ms per step, launches, clocks)."""
            ctx.profile(True)
            l0 = ctx.launches
            tot = 0.0
            with ClockSampler(local, rank == 0) as cs:
                for _ in range(steps):
                    ctx.flush_l2()        # evict the index between timed steps (the 256-term one is about L2-sized)
                    barrier()
                    ctx.timer_start()
                    step()
                    tot += max_over_ranks(ctx.timer_stop())
            tk, tkn = ctx.profile_read("topk")
            mg, mgn = ctx.profile_read("merge")
            ctx.profile(False)
            return tot / steps, tk / max(tkn, 1), mg / max(mgn, 1), ctx.launches - l0 - steps, cs.summary()

        for _ in range(args.warmup):
            bm25_step()
        barrier()
        # headline: shipped configuration (block-max pruning on: lead mode for pairs whose long list can be probed)
        bm_ms, tk_ms, mg_ms, bm_launches, clocks2 = timed_bm25(bm25_step, args.steps, "default")
        if args.dump_outputs:
            ctx.sync()
            bm25_keys = keys.cpu().numpy()     # the last timed step's top-k keys, before later legs overwrite them
        hits_p, n_p, tot_pruned = [x.copy() for x in batch.run_host()] if dist is None else (None, None, None)   # run_host reuses its buffers
        # roofline leg: the same batch with pruning off -- every list of every query is decoded, so the touched bytes
        # are exactly the lists' encoded bytes (what the numerator claims)
        ctx.set_wand(0)
        bm25_step()
        ex_ms, ex_tk_ms, _, _, _ = timed_bm25(bm25_step, max(3, args.steps // 2), "exhaustive")
        hits, n_out, total = [x.copy() for x in batch.run_host()] if dist is None else (None, None, None)
        ctx.set_wand(2)
        seen_pct = None if dist is not None else round(100.0 * float(tot_pruned.sum()) / float(total.sum()), 1)
        if dist is None:   # pruning must not change a single hit (wand differential, over the whole batch)
            assert np.array_equal(n_p, n_out) and np.array_equal(hits_p["doc"], hits["doc"]) and np.array_equal(hits_p["score"], hits["score"])
        # e2e: host query descriptors in, host hits out (index resident: staged at index-load time)
        batch.run_host()
        barrier()
        ctx.timer_start()
        e_steps2 = args.steps
        for _ in range(e_steps2):
            if dist is None:
                hits, n_out, total_e = batch.run_host()
            else:
                hits, n_out = bm25_step(to_host=True)
        be_ms = max_over_ranks(ctx.timer_stop()) / e_steps2
        barrier()
        ex_ach = alg_bytes / (ex_tk_ms * 1e-3) / 1e9
        bm = {
            "metric": "BM25 top-1000, 2-term OR batch: postings of the queried lists per second (BASELINE.json configs[2])",
            "value": round(world * postings / (bm_ms * 1e-3) / 1e6, 1), "unit": "Mdocs/s", "ms_per_step": round(bm_ms, 3),
            "corpus_docs_per_s_M": round(world * n_docs * nq / (bm_ms * 1e-3) / 1e6, 1),
            "config": {"workload": "bm25: %d docs/GPU synthetic Zipf corpus, %d two-term OR queries/step over %d terms, top-%d, block-max "
                                   "pruning on (MaxScore lead mode: pairs whose long list's bound falls below the running threshold stream "
                                   "the short list and probe the long one; everything else is merged exhaustively)" % (n_docs, nq, N_TERMS, TOPK),
                       "postings_per_step": postings, "docs_seen_pct_with_pruning": seen_pct,
                       "exhaustive_ms_per_step": round(ex_ms, 3),
                       "merge": "none" if world == 1 else ("1 NCCL all-gather per step, enqueued by libsdbg.so on the scan's stream" if via_c
                                                         else "torch.distributed all-gather (fallback)"),
                       "l2": "256 MB write between timed steps (index ~L2-sized)"},
            "e2e": {"value": round(world * postings / (be_ms * 1e-3) / 1e6, 1), "unit": "Mdocs/s",
                    "h2d_bytes_per_step": int(len(batch.off) * 4 + (len(batch.off) - 1) * 2 * 32),
                    "d2h_bytes_per_step": nq * TOPK * 8 + nq * 12, "ms_per_step": round(be_ms, 3)},
            "gpu_launches": int(bm_launches),
            "roofline": {"bound": "hbm", "achieved": round(ex_ach, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(ex_ach / hbm_peak, 4),
                         "traffic": ncu_traffic("bm25_merge_kernel", n_docs), "kernel": "bm25_merge_kernel<2> (pruning off: every list decoded)",
                         "kernel_ms": round(ex_tk_ms, 3), "merge_kernel_ms": round(mg_ms, 3), "algorithmic_bytes": alg_bytes, "peak_source": peak_src,
                         "note": "touched bytes = encoded doc+freq blocks of both lists of every query + 1 B norm per posting + 12 B per hit; "
                                 "the kernel is bound by instruction issue (see DESIGN.md 4.3), the HBM fraction is reported as asked"},
            "clocks": clocks2,
        }
        clocks = merge_clocks(clocks, clocks2)
        line["clocks"] = clocks
        # ---- second workload: an index far larger than L2 (4096 terms with a flat tail), pruning off ----
        if world == 1 and not args.skip_extra:
            hn = 4096
            hseg = sdb.Segment(ctx, n_docs)
            hdc, hsum = hseg.synth_corpus(0, 0, hn, threads=min(cores, 64), p_floor=0.004)
            hreader = sdb.IndexReader([hseg], n_docs, hsum, hdc)
            hq = make_queries(args.queries, n_terms=hn, stream=9)[1:] + [[7, 4000]]
            hb = sdb.PreparedBatch(hreader, hq, sdb.OR, scorer, TOPK)
            hp = int(sum(int(hdc[a]) + int(hdc[b]) for a, b in hq))
            htb = hseg.term_bytes(hn)
            h_alg = int(sum(int(htb[a]) + int(htb[b]) + int(hdc[a]) + int(hdc[b]) for a, b in hq)) + len(hq) * TOPK * 12
            ctx.set_wand(0)
            hkeys = torch.zeros(len(hq) * TOPK, dtype=torch.int64, device=dev)
            hstep = lambda: hb.run_device(0, hkeys.data_ptr())
            hstep()
            h_ms, h_tk, _, _, _ = timed_bm25(hstep, 3, "hbm")
            # parity of this workload: the new kernels against the round-1 window kernel, bit for bit, on a sample
            sample = hq[:64]
            s_new = sdb.ExecuteTopKBatch(hreader, sample, sdb.OR, scorer, TOPK)
            os.environ["SDBG_STREAM"] = "0"
            s_old = sdb.ExecuteTopKBatch(hreader, sample, sdb.OR, scorer, TOPK)
            os.environ.pop("SDBG_STREAM", None)
            assert np.array_equal(s_new[0]["doc"], s_old[0]["doc"]) and np.array_equal(s_new[0]["score"], s_old[0]["score"]) and np.array_equal(s_new[2], s_old[2])
            ctx.set_wand(2)
            index_bytes = int(sum(int(x) for x in htb)) + int(sum(int(x) for x in hdc))
            bm["roofline_hbm_resident"] = {
                "workload": "%d terms (Zipf head, inclusion probability floored at 0.004): %.0f MB of posting blocks, %d two-term OR queries, pruning off"
                            % (hn, index_bytes / 1e6, len(hq)),
                "value": round(hp / (h_ms * 1e-3) / 1e6, 1), "unit": "Mdocs/s", "ms_per_step": round(h_ms, 3), "kernel_ms": round(h_tk, 3),
                "achieved": round(h_alg / (h_tk * 1e-3) / 1e9, 1), "peak": hbm_peak, "frac": round(h_alg / (h_tk * 1e-3) / 1e9 / hbm_peak, 4),
                "algorithmic_bytes": h_alg, "parity": "64 sampled queries bit-exact against the round-1 window kernel"}
            hseg.close()
        if rank == 0 and world == 1 and not args.skip_cpu:
            oseg, odc, osdl = cpu_bm25_setup(n_docs, threads)
            assert np.array_equal(odc, dc) and osdl == sum_dl
            cq = queries[: max(args.cpu_queries, 256)]
            dt, ohits, on, scored = cpu_bm25(oseg, odc, osdl, n_docs, cq, threads, mode=2)
            cp = sum(int(dc[a]) + int(dc[b]) for a, b in cq)
            bm["cpu_baseline"] = {"value": round(cp / dt / 1e6, 2), "unit": "Mdocs/s", "cores": threads, "kind": "port",
                                  "sample": "%d of the %d queries, block-max pruned oracle (scored %.0f%% of postings), simdcomp unpack via oracle/_ref"
                                            % (len(cq), nq, 100.0 * scored / max(cp, 1))}
            # full-size parity of this run against the CPU oracle: every sampled query, docs and fp32 score bits
            for qi in range(len(cq)):
                n = int(on[qi])
                assert int(n_out[qi]) == n, "bm25 parity (count) q%d" % qi
                assert np.array_equal(hits[qi, :n]["doc"], ohits[qi, :n]["doc"]), "bm25 parity (docs) q%d" % qi
                assert np.array_equal(hits[qi, :n]["score"], ohits[qi, :n]["score"]), "bm25 parity (scores) q%d" % qi
            bm["config"]["parity"] = "%d queries of this run bit-exact (docs, order, fp32 score bits) against the CPU oracle; pruned == exhaustive over all %d" % (len(cq), nq)
        line["bm25"] = bm
        line["gpu_launches"] = int(gb_launches + bm_launches)
    # ------------------------------------------------------------------ BASELINE configs[0] and configs[3] (N=1)
    if world == 1 and not args.skip_extra and not args.skip_bm25:
        import orc
        other = {}
        # configs[0]: 1 Mi rows int64 + float64, single filter + COUNT/SUM; reference CPU path on ONE thread
        r1 = 1 << 20
        s1 = sdb.Segment(ctx, r1)
        s1.synth_column(1, 21, 1, 0, r1)   # x = h % 1e6
        s1.synth_column(2, 22, 2, 0, r1)   # y in [0,1)
        sc1 = sdb.IResearchScan([s1])
        q_int = ([sdb.pred(1, "LT", 250000)], 1)
        q_flt = ([sdb.pred(2, "LT", 0.25)], 2)
        run_int, run_flt = sc1.prepare_count_sum(*q_int), sc1.prepare_count_sum(*q_flt)   # arguments marshalled once
        for _ in range(5):
            run_int(); run_flt()
        reps = 200
        ctx.sync()
        t = time.perf_counter()
        for _ in range(reps):
            g_int = run_int(); g_flt = run_flt()
        ms1 = (time.perf_counter() - t) * 1e3 / (2 * reps)      # host wall clock per call: the result is on the host when it returns
        assert g_int == sc1.count_sum(*q_int) and g_flt[:2] == sc1.count_sum(*q_flt)[:2]
        o1 = orc.Segment(r1, has_wand=False)
        o1.add_column(1, orc.synth_column(21, 1, 0, r1)); o1.add_column(2, orc.synth_column(22, 2, 0, r1))
        t = time.perf_counter()
        for _ in range(5):
            c_int = orc.filter_count_sum([o1], [orc.make_pred(1, "LT", 250000)], 1, threads=1)
            c_flt = orc.filter_count_sum([o1], [orc.make_pred(2, "LT", 0.25, is_float=True)], 2, threads=1)
        cpu1 = (time.perf_counter() - t) / 10
        assert g_int[:2] == c_int[:2] and g_flt[0] == c_flt[0] and abs(g_flt[2] - c_flt[2]) <= 1e-9 * abs(c_flt[2])
        other["configs[0]"] = {"workload": "1 Mi rows, WHERE x<250000 / y<0.25 -> COUNT(*), SUM; host wall clock per C-ABI call, result in host memory on return (launch-bound: 8 MiB)",
                               "value": round(r1 / (ms1 * 1e-3) / 1e6, 1), "unit": "Mrows/s", "us_per_query": round(ms1 * 1e3, 1),
                               "cpu_baseline": {"value": round(r1 / cpu1 / 1e6, 1), "unit": "Mrows/s", "cores": 1, "kind": "port"}}
        s1.close()
        # zonemap skip (DESIGN 4.1): the configs[1] table plus a clustered int64 column ts = row / 100 (an insertion timestamp);
        # WHERE ts BETWEEN lo AND hi keeps 1 % of the rows -> GROUP BY k SUM(v), AVG(w), COUNT(*). Dead 2048-row blocks are never
        # copied, so the bytes read per table row fall far below the 32 B/row of the four referenced columns.
        TS = 20
        seg.synth_column(TS, 0, 7, row0, rows)
        ts_lo = (row0 + rows // 2) // 100
        zp = [sdb.pred(TS, "BETWEEN", ts_lo, ts_lo + rows // 10000 - 1)]
        zres = {}
        for zm in ("1", "0"):
            os.environ["SDBG_ZONEMAP"] = zm
            scan.groupby_partial(zp, K, key_min, span, V, W_, d_i64.data_ptr(), d_f64.data_ptr())
            ctx.sync(); ctx.timer_start()
            for _ in range(10):
                scan.groupby_partial(zp, K, key_min, span, V, W_, d_i64.data_ptr(), d_f64.data_ptr())
            zms = ctx.timer_stop() / 10
            zres[zm] = (zms, ctx.scan_stats(), scan.groupby_finalize(key_min, span, d_i64.data_ptr(), d_f64.data_ptr(), span))
        os.environ.pop("SDBG_ZONEMAP", None)
        (z_on, (zb, zs), zr_on), (z_off, _, zr_off) = zres["1"], zres["0"]
        for fld in ("key", "count", "sum_lo", "sum_hi", "cnt_f64"):
            assert np.array_equal(zr_on[fld], zr_off[fld]), fld
        assert np.allclose(zr_on["sum_f64"], zr_off["sum_f64"], rtol=1e-12, atol=0) and int(zr_on["count"].sum()) == rows // 100   # SUM(double) REDs land in arbitrary order
        other["zonemap"] = {"workload": "%d rows x 4 referenced columns (32 B/row), WHERE ts BETWEEN .. (1 %% of rows, clustered column) -> GROUP BY k SUM(v), AVG(w), COUNT(*)" % rows,
                            "value": round(rows / (z_on * 1e-3) / 1e6, 1), "unit": "Mrows/s", "ms_per_step": round(z_on, 4),
                            "ms_per_step_without_zonemaps": round(z_off, 4), "blocks": int(zb), "blocks_skipped": int(zs),
                            "bytes_read_per_row": round(32.0 * (zb - zs) / max(zb, 1), 3), "parity": "groups identical with and without the skip (SUM(double) to 1e-12: RED order)"}
        # configs[3]: 5-term conjunctive BM25 + range filter on an int32 INCLUDE column, top-1000 (hybrid). The five
        # terms have p = 0.50, 0.40, 0.30, 0.25, 0.20 (SURVEY §8d: 16.5 M postings, ~30 k conjunctive matches); they live in
        # a segment of their own over the same docs (generator terms 1000000..1000004).
        T4 = 1000000
        seg4 = sdb.Segment(ctx, n_docs)
        dc4, sum_dl4 = seg4.synth_corpus(rank * n_docs, T4, 5, threads=min(cores, 64))
        assert sum_dl4 == sum_dl
        seg4.synth_column(9, 2, 6, rank * n_docs + 1, n_docs)   # n = h % 1e6 for docs 1..N
        reader4 = sdb.IndexReader([seg4], n_docs, sum_dl4, dc4)
        filt = sdb.pred(9, "BETWEEN", 250000, 749999)
        q4 = [0, 1, 2, 3, 4]
        nq4 = 64
        b4 = sdb.PreparedBatch(reader4, [q4] * nq4, sdb.AND, scorer, TOPK, filt=filt)
        b4.run_host()
        ctx.flush_l2(); ctx.sync(); ctx.timer_start()
        h4, n4, t4 = b4.run_host()
        ms4 = ctx.timer_stop()
        p4 = int(sum(int(dc4[t]) for t in q4))
        oseg4, odc4, osdl4 = orc.synth_segment_mt(n_docs, T4, 5, doc0=0, threads=threads)
        assert np.array_equal(odc4, dc4)
        col = np.zeros(n_docs, np.int32)
        col[:] = orc.synth_column(2, 1, 1, n_docs).astype(np.int32)
        oseg4.add_column(9, col)
        qt4 = []
        for t_ in q4:
            st = orc.bm25_stats(n_docs, sum_dl, int(dc4[t_]))
            x = orc.BM25Term(); x.idf, x.norm_const, x.norm_length, x.boost, x.term = st.idf, st.norm_const, st.norm_length, 1.0, t_
            qt4.append(x)
        ncpu4 = min(threads, 32)
        tcpu = time.perf_counter()
        oh4, on4, ot4, _ = orc.bm25_topk_batch([oseg4], "AND", [qt4] * ncpu4, TOPK, filt=orc.make_pred(9, "BETWEEN", 250000, 749999), mode=1, threads=threads)
        cpu4 = time.perf_counter() - tcpu
        assert np.array_equal(h4[0, :n4[0]]["doc"], oh4[0, :on4[0]]["doc"]) and np.array_equal(h4[0, :n4[0]]["score"], oh4[0, :on4[0]]["score"])
        assert int(t4[0]) == int(ot4[0])
        other["configs[3]"] = {"workload": "%d docs, 5-term AND (p = .5/.4/.3/.25/.2: %d postings) + n BETWEEN 250000 AND 749999, top-1000; batch of %d, host call; "
                                           "shortest list streamed, the other four probed per candidate (lead list + LazySeek)" % (n_docs, p4, nq4),
                               "value": round(nq4 * p4 / (ms4 * 1e-3) / 1e6, 1), "unit": "Mdocs/s", "ms_per_query": round(ms4 / nq4, 3), "matches": int(t4[0]),
                               "cpu_baseline": {"value": round(ncpu4 * p4 / cpu4 / 1e6, 1), "unit": "Mdocs/s", "cores": min(threads, ncpu4), "kind": "port",
                                                "sample": "%d concurrent copies of the query" % ncpu4}}
        seg4.close()
        line["other_configs"] = other
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, bm25_keys, nq)
    if rank == 0:
        emit_line(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
