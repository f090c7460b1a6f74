#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native MyScaleDB hot path.

Workload (BASELINE.json configs[1], the largest single-GPU configuration):
    FLAT brute-force inner product, 10M x 768-d bf16 corpus, batch of 1024 queries, top-10.
One "step" = one query batch scanned against the whole (sharded) corpus.
  value : QPS with corpus AND queries resident in HBM (device-timed, CUDA events)
  e2e   : QPS through the C-ABI host call b200_corpus_search(): pinned host queries in,
          host results out, H2D/D2H inside the timed region.  The corpus is index state
          (loaded once, like VICacheManager keeps a FLAT index resident); its upload is not a
          per-step input.
Multi-GPU (--gpus N, launched by torch.distributed.run): the 10M rows are sharded N ways
(strong scaling, total work fixed), every rank scans its shard, one NCCL all-gather of the
per-shard top-k, one merge kernel.
--impl reference: the CPU arm -- the oracle's restatement of the reference's brute-force path
(one thread per part, SIMD inner-product blocks; the reference binary cannot be built here,
see DESIGN.md), timed on a bounded row sample and scaled linearly to the full corpus.
--dump-outputs DIR: the answer of the last timed step (what a caller of the timed path receives) as DIR/distances.npy
(float32) and DIR/ids.npy (float64), so that two builds can be compared output for output on identical seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

# BASELINE.json's metric ("QPS @ recall@10>=0.95 ...") on configs[1]; exact brute force, so recall@10 is 1.0
METRIC = "QPS @ recall@10>=0.95 (exact: recall 1.0), FLAT brute-force IP top-10, 10M x 768-d bf16, batch 1024"


def metric_name(a):
    rows = f"{a.rows // 1_000_000}M" if a.rows % 1_000_000 == 0 else str(a.rows)
    return f"QPS @ recall@10>=0.95 (exact: recall 1.0), FLAT brute-force IP top-{a.k}, {rows} x {a.dim}-d bf16, batch {a.nq}"
CHUNK = 250_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--nq", type=int, default=1024)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU-baseline sample duration")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="A/B runs: skip verification and the extra keys")
    ap.add_argument("--index-rows", type=int, default=100_000_000, help="rows of the MSTG-class index extra (BASELINE configs[2]); 0 = skip")
    ap.add_argument("--index-nq", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's distances and ids as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times the CPU oracle on a row sample)")
    return a


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, dis, ids):
    """Writes the top-k answer as float32 distances / float64 ids (exact below 2**53).  Above DUMP_BYTES, a fixed seeded
    sample of query rows is written, with their indices in query_rows.npy."""
    import numpy as np
    nq = dis.shape[0]
    cap = max(1, DUMP_BYTES // max(1, dis.shape[1] * (4 + 8)))
    arrays = {}
    if nq > cap:
        rows = np.sort(np.random.default_rng(0).choice(nq, size=cap, replace=False))
        dis, ids = dis[rows], ids[rows]
        arrays["query_rows"] = rows.astype(np.float64)
    arrays["distances"] = np.ascontiguousarray(dis, dtype=np.float32)
    arrays["ids"] = np.ascontiguousarray(ids, dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def config_of(a, n):
    return {"workload": f"FLAT brute-force IP, {a.rows} x {a.dim}-d bf16, batch {a.nq} queries, top-{a.k} "
                        + ("(BASELINE.json configs[1])" if (a.rows, a.dim, a.nq, a.k) == (10_000_000, 768, 1024, 10) else "(non-default size)"),
            "rows": a.rows, "dim": a.dim, "batch_queries": a.nq, "k": a.k,
            "sharding": (f"rows/{n} per GPU; b200_sharded_corpus_search(): tensor-core scan -> one ncclAllGather of the packed per-shard "
                         "top-k -> merge kernel, replayed as one CUDA graph per step") if n > 1 else "single GPU",
            "cache": f"inputs ({a.rows * a.dim * 2 / n / 1e9:.1f} GB of corpus rows per GPU) larger than the 126 MB L2; no flush needed"}


_NVML_LOOP = r"""
import sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
print("ready", mx, flush=True)
while True:
    print(time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), int(get(h)), flush=True)
    time.sleep(0.004)
"""


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region: a helper process polls NVML every ~5 ms
    (a thread in this process starves behind the launch loop's GIL; nvidia-smi -lms is too coarse)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        self.phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
        self.proc, self.max_mhz, self.t0, self.t1 = None, None, None, None

    def launch(self):
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", _NVML_LOOP, str(self.phys)], stdout=subprocess.PIPE, text=True)
            first = self.proc.stdout.readline().split()
            self.max_mhz = float(first[1]) if first and first[0] == "ready" else None
        except Exception:
            self.proc = None

    def start(self):
        if self.proc is None:
            self.launch()
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML helper unavailable"], "samples": 0}
        time.sleep(0.02)
        self.proc.terminate()
        out = self.proc.stdout.read()
        sm, mask = [], 0
        for ln in out.splitlines():
            f = ln.split()
            if len(f) == 3:
                try:
                    t, c, r = float(f[0]), float(f[1]), int(f[2])
                except ValueError:
                    continue
                if self.t0 <= t <= self.t1:
                    sm.append(c)
                    mask |= r
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples in the timed region"], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for bit, n in self.REASONS.items() if mask & bit), "samples": len(sm),
                "how": "NVML helper process, ~5 ms period, samples inside the timed region only"}


def make_queries(a):
    import torch
    g = torch.Generator(device="cpu"); g.manual_seed(4)
    q = torch.randn((a.nq, a.dim), generator=g, dtype=torch.float32)
    return q.to(torch.bfloat16).to(torch.float32)  # bf16-valued fp32, the GEMM path's input contract


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _cpu_sample_data(a, rows):
    import torch
    g = torch.Generator(device="cpu"); g.manual_seed(1000)
    y = torch.randn((rows, a.dim), generator=g, dtype=torch.float32).to(torch.bfloat16).to(torch.float32).numpy()
    return make_queries(a).numpy(), y


def _cpu_child(conn, a_dict, rows, threads, use_blas, reps):
    """Runs in a spawned child: a crash inside a BLAS thread pool must not take the bench down."""
    import argparse as _ap
    a = _ap.Namespace(**a_dict)
    import oracle as orc
    q, y = _cpu_sample_data(a, rows)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        if use_blas:
            if orc.knn_flat_parts_blas(orc.IP, q, y, a.k, threads) is None:
                conn.send(None)
                return
        else:
            orc.knn_flat_parts(orc.IP, q, y, a.k, threads)
        ts.append(time.perf_counter() - t0)
    conn.send(ts)


def run_cpu_sample(a, rows, threads, use_blas, reps=1, timeout=600):
    """Times the oracle's threaded brute force (the reference's CPU algorithm) on `rows` corpus rows.
    Returns the list of per-repetition seconds, or None if the child failed."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    parent, child = ctx.Pipe()
    p = ctx.Process(target=_cpu_child, args=(child, vars(a), rows, threads, use_blas, reps))
    p.start()
    res = parent.recv() if parent.poll(timeout) else None
    p.join(10)
    if p.is_alive():
        p.kill()
    return res if p.exitcode == 0 else None


def cpu_plan(a, budget_s):
    """Pick (use_blas, threads, rows): Faiss BLAS form if OpenBLAS works here, sample sized to budget_s."""
    logical = cpu_threads()
    for use_blas, threads in ((True, min(logical, 64)), (False, logical)):   # OpenBLAS: <= 64 concurrent callers
        probe_rows = 2048 * max(1, threads // 8)
        ts = run_cpu_sample(a, probe_rows, threads, use_blas, reps=2, timeout=300)
        if ts:
            rate = probe_rows / max(min(ts), 1e-6)
            rows = int(min(a.rows, 2_000_000, max(probe_rows, rate * budget_s)))
            return use_blas, threads, rows
    raise RuntimeError("CPU baseline could not run")


def cpu_baseline(a):
    use_blas, threads, rows = cpu_plan(a, a.cpu_seconds)
    t = run_cpu_sample(a, rows, threads, use_blas, reps=1)[0]
    qps = a.nq / (t * (a.rows / rows))
    how = ("one single-threaded OpenBLAS sgemm stream per part (Faiss BLAS form)" if use_blas
           else "one thread per part, portable SIMD inner-product blocks")
    return {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
            "sample": f"{a.nq} queries x {rows} of {a.rows} rows (bf16-valued fp32), {t:.2f} s on {threads} threads, {how}; "
                      f"oracle/cpu_baseline.c; scaled linearly to {a.rows} rows"}


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = 150.0 / max(1, a.steps + a.warmup)            # keep the whole arm within a few minutes
    use_blas, threads, rows = cpu_plan(a, min(a.cpu_seconds, budget))
    ts = run_cpu_sample(a, rows, threads, use_blas, reps=a.warmup + a.steps, timeout=900)[a.warmup:]
    t_step = sum(ts) / len(ts) * (a.rows / rows)
    qps = a.nq / t_step
    how = ("one single-threaded OpenBLAS sgemm stream per part (Faiss BLAS form)" if use_blas
           else "one thread per part, portable SIMD inner-product blocks")
    cb = {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
          "sample": f"each step = {a.nq} queries x {rows} of {a.rows} rows, scaled linearly; oracle/cpu_baseline.c, {how} "
                    "(reference threading model: ThreadPool over parts, kernel single-threaded inside a part)"}
    print(json.dumps({"impl": "reference", "metric": metric_name(a), "value": qps, "unit": "queries/s", "n_gpus": a.gpus,
                      "steps": a.steps, "warmup": a.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True,
                      "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": config_of(a, a.gpus), "cpu_baseline": cb,
                      "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def _agree(d_a, i_a, d_b, i_b, rtol):
    """Two top-k answers of the same queries agree: distances elementwise within rtol, ids identical except where two
    candidates are closer than the tolerance (a swap of near ties or a different pick at the k-th boundary)."""
    import numpy as np
    scale = np.maximum(np.abs(d_b), 1.0)
    err = float((np.abs(d_a - d_b) / scale).max())
    if err > rtol:
        return False, err, 0.0
    same = i_a == i_b
    for q, j in np.argwhere(~same):
        hit = np.flatnonzero(i_b[q] == i_a[q, j])
        ref = d_b[q, hit[0]] if hit.size else d_b[q, -1]
        if abs(d_a[q, j] - ref) > rtol * max(1.0, abs(ref)):
            return False, err, float(same.mean())
    return True, err, float(same.mean())


def verify_results(a, index, corpus, q_host, q_dev, d_res, i_res, row0, shard_rows, N, rank, dev):
    """(1) 16 sampled queries re-answered by the fp32 FMA scan kernel (path 1, an independent kernel) over every shard
    and merged on the host; (2) 2 of them re-answered by the CPU oracle over the full corpus (rows read back from HBM).
    Both must agree with what the timed tensor-core path (+ all-gather + merge kernel at N > 1) returned."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import oracle as orc
    k, nq = a.k, a.nq
    rng = np.random.default_rng(12345)
    sample = np.sort(rng.choice(nq, size=min(16, nq), replace=False))
    qs = q_dev[torch.as_tensor(sample, device=dev)].contiguous()
    sd = torch.empty((len(sample), k), dtype=torch.float32, device=dev)
    si = torch.empty((len(sample), k), dtype=torch.int64, device=dev)
    index.set_path(1)
    index.search_device(qs.data_ptr(), len(sample), k, sd.data_ptr(), si.data_ptr(), id_offset=row0,
                        stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    index.set_path(0)
    # CPU oracle on 2 of the sampled queries over this rank's rows
    two = sample[:2]
    xq = np.ascontiguousarray(q_host.numpy()[two])
    od = np.full((len(two), 0), 0, np.float32); oi = np.zeros((len(two), 0), np.int64)
    for off in range(0, shard_rows, 500_000):
        m = min(500_000, shard_rows - off)
        rows = corpus[off:off + m].to(torch.float32).cpu().numpy()
        cd, ci = orc.knn_flat(orc.IP, xq, rows, k)
        od = np.concatenate([od, cd], axis=1); oi = np.concatenate([oi, np.where(ci >= 0, ci + row0 + off, -1)], axis=1)
    cpu_d = torch.tensor(od, device=dev); cpu_i = torch.tensor(oi, device=dev)
    if N > 1:
        def gather(t):
            parts = [torch.empty_like(t) for _ in range(N)]
            dist.all_gather(parts, t.contiguous())
            return torch.cat(parts, dim=1)
        # every rank holds the same number of chunk candidates only if shards are equal: pad to the max width
        width = torch.tensor([cpu_d.shape[1]], device=dev); dist.all_reduce(width, op=dist.ReduceOp.MAX)
        pad = int(width.item()) - cpu_d.shape[1]
        if pad:
            cpu_d = torch.cat([cpu_d, torch.full((cpu_d.shape[0], pad), -3e38, device=dev)], dim=1)
            cpu_i = torch.cat([cpu_i, torch.full((cpu_i.shape[0], pad), -1, device=dev, dtype=torch.int64)], dim=1)
        sd, si, cpu_d, cpu_i = gather(sd), gather(si), gather(cpu_d), gather(cpu_i)

    def host_topk(d, i):
        d, i = d.cpu().numpy(), i.cpu().numpy()
        out_d = np.empty((d.shape[0], k), np.float32); out_i = np.empty((d.shape[0], k), np.int64)
        for q in range(d.shape[0]):
            ok = i[q] >= 0
            order = np.lexsort((i[q][ok], -d[q][ok]))[:k]
            out_d[q], out_i[q] = d[q][ok][order], i[q][ok][order]
        return out_d, out_i
    scan_d, scan_i = host_topk(sd, si)
    cpu_d, cpu_i = host_topk(cpu_d, cpu_i)
    ok1, err1, same1 = _agree(d_res[sample], i_res[sample], scan_d, scan_i, 2e-4)
    ok2, err2, same2 = _agree(d_res[two], i_res[two], cpu_d, cpu_i, 2e-4)
    if not (ok1 and ok2):
        raise AssertionError(f"timed path disagrees with its checkers: scan kernel ok={ok1} (max rel err {err1:.2e}, ids "
                             f"{same1:.3f}), CPU oracle ok={ok2} (max rel err {err2:.2e}, ids {same2:.3f})")
    return {"scan_kernel_queries": int(len(sample)), "scan_kernel_ids_identical": same1, "scan_kernel_max_rel_err": err1,
            "cpu_oracle_queries": int(len(two)), "cpu_oracle_ids_identical": same2, "cpu_oracle_max_rel_err": err2,
            "rows_checked": a.rows, "shards": N,
            "what": "results of the timed path (tensor-core top-k" + (", NCCL all-gather, merge kernel" if N > 1 else "")
                    + ") vs the fp32 scan kernel over every shard merged on the host, and vs oracle/vs_oracle.c over all rows"}


def traffic_from_profile(a, n_gpus):
    """DRAM bytes per launch of the headline kernel on THIS workload from the committed ncu capture, or None."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "gemm_topk_traffic.json")))
        w = rec["workload"]
        if n_gpus == 1 and (w["rows"], w["dim"], w["nq"], w["k"]) == (a.rows, a.dim, a.nq, a.k):
            return rec["dram_bytes_read"] + rec["dram_bytes_write"]
    except Exception:
        pass
    return None


def latency_extra():
    """BASELINE configs[0]: FLAT L2 distance(), 10k x 128 fp32, ONE query, top-10, a part resident in HBM: median latency of
    the C-ABI host call (single fused launch) next to the reference's CPU form on one core (faiss nx < 20: exact differences,
    AVX-512 through target_clones; one thread per part, VIWithDataPart.h:350)."""
    import numpy as np

    import myscaledb_b200 as b2
    import oracle as orc
    rng = np.random.default_rng(1)
    y = rng.standard_normal((10_000, 128)).astype(np.float32)
    x = rng.standard_normal((1, 128)).astype(np.float32)
    c = b2.Corpus(b2.L2, 128).append(y)
    dg, ig = c.search(x, 10)
    do, io = orc.knn_flat(orc.L2, x, y, 10)
    ok = bool((ig == io).all() and np.allclose(dg, do, rtol=1e-4))

    def med(fn, reps, warm):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
        ts.sort()
        return ts[len(ts) // 2] * 1e6
    gpu_us = med(lambda: c.search(x, 10), 300, 30)
    one_shot_us = med(lambda: b2.part_scan(b2.L2, x, y, 10), 50, 5)
    cpu_us = med(lambda: orc.knn_flat_simd(orc.L2, x, y, 10), 50, 3)
    c.close()
    return {"workload": "FLAT L2 distance(), 10k x 128 fp32, 1 query, top-10 (BASELINE.json configs[0])", "matches_oracle": ok,
            "resident_call_us": round(gpu_us, 1), "one_shot_part_scan_us": round(one_shot_us, 1),
            "cpu_simd_one_core_us": round(cpu_us, 1), "bytes_per_query": 10_000 * 128 * 4,
            "note": "resident = b200_corpus_search() on a part kept in HBM (one fused launch, query and result through mapped pinned "
                    "memory); one_shot = b200_part_scan() including the H2D of the 5 MB part; cpu = oracle/cpu_baseline.c "
                    "orc_knn_flat_simd (AVX-512, one thread per part like the reference)"}


def index_extra(a, dev, N, rank, comm):
    """BASELINE configs[2] / the metric's own scale: MSTG-class index, 100 M x 768 fp32 clustered rows (SURVEY 8d: 10 000 Gaussian
    centres, points = centre + N(0, 0.3^2)), batch of 256 queries, top-10, rows sharded over the N GPUs.  Rows are generated
    chunk by chunk in HBM and streamed into b200_index_add_device (bf16 lists; the fp32 rows are not kept: 307 GB);
    ground truth = exact fp32 scan of the regenerated chunks; the sharded search is b200_sharded_index_search."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import myscaledb_b200 as b2
    from myscaledb_b200.sharding import shard_range
    CH = 500_000
    rows = a.index_rows
    free_b = torch.cuda.mem_get_info()[0]
    per_row = a.dim * 2 + 16
    cap = int(free_b * 0.88 / per_row / CH) * CH * N
    if rows > cap:
        rows = cap
    rows = (rows // (CH * N)) * CH * N
    if rows <= 0:
        return {"error": "not enough free HBM for the index extra"}
    r0, r1 = shard_range(rows, N, rank, CH)
    shard = r1 - r0
    g = torch.Generator(device=dev); g.manual_seed(5)
    centres = torch.randn((10_000, a.dim), generator=g, device=dev)

    def chunk(ci, m, seed_base):
        gg = torch.Generator(device=dev); gg.manual_seed(seed_base + ci)
        x = torch.randn((m, a.dim), generator=gg, device=dev)
        idx = torch.randint(0, 10_000, (m,), generator=gg, device=dev)
        return (centres[idx] + 0.3 * x).contiguous()
    nlist = 16384 if shard >= 4_000_000 else max(256, int(4 * shard ** 0.5))
    t0 = time.perf_counter()
    ix = b2.VectorIndex("MSTG", b2.L2, a.dim, f"ncentroids={nlist}, keep_raw=0")
    ix.reserve(shard)
    n_chunks = shard // CH
    per = -(-min(shard, 64 * nlist) // n_chunks)
    parts = []
    for i in range(n_chunks):   # a strided slice is a VIEW of its 1.4 GB chunk: copy it out, drop the chunk
        x = chunk((r0 // CH) + i, CH, 100)
        parts.append(x[:: max(1, CH // per)][:per].clone())
        del x
    sample = torch.cat(parts).contiguous()
    del parts
    torch.cuda.synchronize()
    ix.train_device(sample.data_ptr(), sample.shape[0])
    del sample
    for i in range(n_chunks):
        x = chunk((r0 // CH) + i, CH, 100)
        torch.cuda.synchronize()
        ix.add_device(x.data_ptr(), CH)
        del x
    ix.finalize()
    build_s = time.perf_counter() - t0
    nq, k = a.index_nq, a.k
    q = chunk(0, nq, 6_000_000)
    # ---- ground truth: exact fp32 scan of every regenerated chunk (3xTF32 tensor-core kernel), merged over chunks and ranks
    nt = min(nq, 128)
    t0 = time.perf_counter()
    od = torch.empty((nt, k), dtype=torch.float32, device=dev); oi = torch.empty((nt, k), dtype=torch.int64, device=dev)
    td = torch.empty((nt, 0), dtype=torch.float32, device=dev); ti = torch.empty((nt, 0), dtype=torch.int64, device=dev)
    s = torch.cuda.current_stream().cuda_stream
    for i in range(n_chunks):
        x = chunk((r0 // CH) + i, CH, 100)
        torch.cuda.synchronize()
        c = b2.Corpus(b2.L2, a.dim)
        c.adopt_device(x.data_ptr(), CH)
        c.search_device(q.data_ptr(), nt, k, od.data_ptr(), oi.data_ptr(), id_offset=r0 + i * CH, stream=s)
        torch.cuda.synchronize()
        c.close()
        td = torch.cat([td, od], 1); ti = torch.cat([ti, oi], 1)
        if td.shape[1] >= 32 * k:
            o = torch.argsort(td, dim=1)[:, :k]
            td, ti = torch.gather(td, 1, o), torch.gather(ti, 1, o)
        del x
    o = torch.argsort(td, dim=1)[:, :k]
    td, ti = torch.gather(td, 1, o).contiguous(), torch.gather(ti, 1, o).contiguous()
    if N > 1:
        gd = [torch.empty_like(td) for _ in range(N)]; gi = [torch.empty_like(ti) for _ in range(N)]
        dist.all_gather(gd, td); dist.all_gather(gi, ti)
        td, ti = torch.cat(gd, 1), torch.cat(gi, 1)
        o = torch.argsort(td, dim=1)[:, :k]
        ti = torch.gather(ti, 1, o)
    truth = ti.cpu().numpy()
    truth_s = time.perf_counter() - t0
    # ---- timed searches
    res_d = torch.empty((nq, k), dtype=torch.float32, device=dev); res_i = torch.empty((nq, k), dtype=torch.int64, device=dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)
    ix.enable_timing(True)
    runs = []
    for nprobe in (1, 2, 4, 8):
        par = f"nprobe={nprobe}"

        def step():
            if N == 1:
                ix.search_device(q.data_ptr(), nq, k, res_d.data_ptr(), res_i.data_ptr(), par, id_offset=r0, stream=s)
            else:
                comm.sharded_index_search(ix, b2.L2, q.data_ptr(), nq, k, par, res_d.data_ptr(), res_i.data_ptr(), r0, s)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        if N > 1:
            dist.barrier()
        ix.last_scan(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            step()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        if N > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        sc = ix.last_scan(reset=True)
        ids = res_i.cpu().numpy()
        rec = float(np.mean([len(set(ids[j].tolist()) & set(truth[j].tolist())) / k for j in range(nt)]))
        kms = sc["kernel_ms"] / max(1, sc["launches"])
        gb = sc["rows_streamed"] * sc["payload_row_bytes"] / 1e9
        runs.append({"nprobe": nprobe, "qps": nq / ms * 1e3, "ms_per_batch": ms, "recall_at_10": rec,
                     "scan_kernel_ms_rank0": kms, "scan_GB_rank0": gb, "scan_GB_per_s_rank0": gb / kms * 1e3 if kms else None,
                     "frac_of_hbm_peak_rank0": gb / kms * 1e3 / hbm if kms else None,
                     "bytes_per_query_all_shards": gb * 1e9 / nq * N, "phase_ms_rank0": ix.phase_ms()})
        if rec >= 0.999:
            break
    good = [r for r in runs if r["recall_at_10"] >= 0.95]
    best = max(good, key=lambda r: r["qps"]) if good else None
    mem = ix.memory_bytes()
    ix.close()
    return {"workload": f"MSTG-class index (paged IVF, bf16 lists, grouped tensor-core scan), {rows} x {a.dim} fp32 clustered rows "
                        f"(10 000 centres, sigma 0.3), batch {nq}, top-{k}, rows sharded over {N} GPU(s) (BASELINE.json configs[2])",
            "rows": rows, "nlist_per_shard": nlist, "build_s_per_shard": build_s, "index_GB_per_shard": mem / 1e9,
            "truth": f"exact fp32 scan of all rows for {nt} queries ({truth_s:.1f} s)",
            "qps_at_recall_0.95": best["qps"] if best else None, "best": best, "runs": runs,
            "hbm_peak_GB_per_s": hbm,
            "note": "QPS device-timed (CUDA events, max over ranks), queries resident; exact brute force over the same rows on the "
                    "tensor cores runs at ~8 k QPS per 100 M rows (round 1, profiles/r01_bench_line_100m_n1.json)"}


def main():
    a = parse()
    if a.impl == "reference":
        return reference_arm(a)

    import numpy as np
    import torch
    import torch.distributed as dist

    import myscaledb_b200 as b2
    from myscaledb_b200 import search as S

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N = world
    assert a.rows % (N * CHUNK) == 0 or N == 1, "rows must split into 250k-row chunks per rank"

    # ---- synthetic corpus shard, generated in HBM (seeded per global 250k-row chunk) ----
    from myscaledb_b200.sharding import shard_range
    row0, row1 = shard_range(a.rows, N, rank, CHUNK)
    shard_rows = row1 - row0
    corpus = torch.empty((shard_rows, a.dim), dtype=torch.bfloat16, device=dev)
    off = 0
    while off < shard_rows:
        m = min(CHUNK, shard_rows - off)
        g = torch.Generator(device=dev); g.manual_seed(1000 + (row0 + off) // CHUNK)
        corpus[off:off + m] = torch.randn((m, a.dim), generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
        off += m
    q_host = make_queries(a).pin_memory()
    q_dev = q_host.to(dev)
    torch.cuda.synchronize()

    index = b2.Corpus(b2.IP, a.dim, dtype=S.BF16)
    index.adopt_device(corpus.data_ptr(), shard_rows)
    # per-launch CUDA events for the roofline at N = 1 (the step is one 12 ms kernel); at N > 1 the step runs as one CUDA
    # graph and the kernel is timed in a separate short loop after the timed region
    index_timing = [N == 1]
    index.enable_timing(index_timing[0])

    k, nq = a.k, a.nq
    # one packed record per rank {float dis[nq*k]; int64 ids[nq*k]} -> a single NCCL all-gather
    rec = nq * k * 12
    packed = torch.empty(rec, dtype=torch.uint8, device=dev)
    gathered = torch.empty(N * rec, dtype=torch.uint8, device=dev)
    o_dis = packed[:nq * k * 4].view(torch.float32).view(nq, k)
    o_ids = packed[nq * k * 4:].view(torch.int64).view(nq, k)
    f_dis = torch.empty((nq, k), dtype=torch.float32, device=dev)
    f_ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    h_dis = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    h_ids = torch.empty((nq, k), dtype=torch.int64).pin_memory()

    # N > 1: the communicator below the C ABI (csrc/comm.cu): shard scan -> ONE ncclAllGather of the packed per-shard
    # top-k -> merge kernel, the whole step replayed as one CUDA graph; Python only carried the 128-byte NCCL id
    comm = None
    if N > 1:
        from myscaledb_b200.sharding import Comm
        comm = Comm.from_torch_distributed(dev)
    side = torch.cuda.Stream(device=dev)   # the sharded steps want a real (non-default) stream

    def step_device():
        if N == 1:
            index.search_device(q_dev.data_ptr(), nq, k, o_dis.data_ptr(), o_ids.data_ptr(), id_offset=row0,
                                stream=torch.cuda.current_stream().cuda_stream)
        else:
            comm.sharded_corpus_search(index, q_dev.data_ptr(), nq, k, f_dis.data_ptr(), f_ids.data_ptr(), row0,
                                       torch.cuda.current_stream().cuda_stream, use_graph=not index_timing[0])

    q_np, hd_np, hi_np = q_host.numpy(), h_dis.numpy(), h_ids.numpy()

    def step_e2e():
        # the reference-facing C-ABI call with host buffers: H2D of the queries, kernels (+ all-gather + merge), D2H of the
        # results and the synchronise are all inside the call
        if N == 1:
            return index.search(q_np, k)
        return comm.sharded_corpus_search_host(index, q_np, k, row0, torch.cuda.current_stream().cuda_stream, use_graph=True,
                                               out=(hd_np, hi_np))

    def barrier():
        if N > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the memory-bound FLAT scan on the same resident shard (BASELINE metric: "brute-force GB/s vs HBM peak"),
    #      measured FIRST, on a cool GPU: after the power-capped GEMM loop the same kernel reads 15-20 % slower
    flat_scan = []
    if (rank == 0 or N > 1) and not a.headline_only:
        try:  # an extra as well: a failure here must not cost the headline line
            index.enable_timing(True)
            for nq_s in (1, 8):
                index.set_path(1)
                for _ in range(3):
                    index.search_device(q_dev.data_ptr(), nq_s, k, o_dis.data_ptr(), o_ids.data_ptr(), id_offset=row0,
                                        stream=torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                index.kernel_time(reset=True)
                reps = 10
                for _ in range(reps):
                    index.search_device(q_dev.data_ptr(), nq_s, k, o_dis.data_ptr(), o_ids.data_ptr(), id_offset=row0,
                                        stream=torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                kms, kn = index.kernel_time(reset=True)
                gbs = shard_rows * a.dim * 2 / (kms / max(kn, 1) * 1e-3) / 1e9
                flat_scan.append({"kernel": "flat_scan_kernel (bf16 rows, fp32 FMA)", "queries_per_pass": nq_s,
                                  "ms_per_launch": kms / max(kn, 1), "GB_per_s": gbs, "bytes_per_launch": shard_rows * a.dim * 2})
        except Exception as e:
            flat_scan = [{"error": f"{type(e).__name__}: {e}"[:300]}]
        index.set_path(0)
        index.enable_timing(index_timing[0])

    # ---- device-resident timing (value) ----
    sampler = ClockSampler(local)
    sampler.launch()
    torch.cuda.set_stream(side)
    for _ in range(max(a.warmup, 3)):
        step_device()
    barrier()
    index.kernel_time(reset=True)
    S.launch_count(reset=True)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        step_device()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = S.launch_count()
    if a.dump_outputs and rank == 0:   # now: the e2e loop and the fp32 extra below reuse these buffers
        dump_outputs(a.dump_outputs, (o_dis if N == 1 else f_dis).cpu().numpy(), (o_ids if N == 1 else f_ids).cpu().numpy())
    kern_ms, kern_n = index.kernel_time(reset=True)
    clocks = sampler.stop()
    if N > 1:  # kernel time for the roofline: a few eager steps with per-launch events, outside the timed region
        index_timing[0] = True
        index.enable_timing(True)
        for _ in range(5):
            step_device()
        torch.cuda.synchronize()
        kern_ms, kern_n = index.kernel_time(reset=True)
        index.enable_timing(False)
        index_timing[0] = False
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if N > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / a.steps
    qps = nq / (ms_step * 1e-3)

    # ---- end-to-end timing through the host API ----
    for _ in range(3):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        res = step_e2e()
    torch.cuda.synchronize()
    te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if N > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_qps = nq / (float(te.item()) / a.steps)

    # ---- fp32 rows (the reference's native column type) on the tensor cores: 3xTF32 split GEMM, same batch, a
    #      2M-row fp32 copy of the shard's head (an extra, not the headline)
    fp32_batch = None
    if N == 1 and rank == 0 and not a.headline_only:
        try:  # an extra: never lose the headline line to it (e.g. no HBM left next to a 100M-row corpus)
            m = int(min(shard_rows, 2_000_000))
            y32 = corpus[:m].to(torch.float32)
            ix32 = b2.Corpus(b2.IP, a.dim)
            ix32.adopt_device(y32.data_ptr(), m)
            ix32.enable_timing(True)
            for _ in range(2):
                ix32.search_device(q_dev.data_ptr(), nq, k, o_dis.data_ptr(), o_ids.data_ptr(),
                                   stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            ix32.kernel_time(reset=True)
            for _ in range(5):
                ix32.search_device(q_dev.data_ptr(), nq, k, o_dis.data_ptr(), o_ids.data_ptr(),
                                   stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            kms3, kn3 = ix32.kernel_time(reset=True)
            per = kms3 / max(kn3, 1)
            fp32_batch = {"kernel": "gemm3_topk_kernel (fp32 rows, 3 x tcgen05.mma.kind::tf32 per k-step, fused top-k)",
                          "rows": m, "batch_queries": nq, "ms_per_launch": per,
                          "effective_fp32_TFLOP_per_s": 2.0 * nq * m * a.dim / (per * 1e-3) / 1e12,
                          "tf32_mma_TFLOP_per_s": 3 * 2.0 * nq * m * a.dim / (per * 1e-3) / 1e12,
                          "qps_scaled_to_workload_rows": nq / (per * 1e-3 * shard_rows / m)}
            ix32.close()
            del y32
        except Exception as e:
            fp32_batch = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- verification of the TIMED path's results (the run fails on a mismatch) ----
    d_res, i_res = res
    verified = None
    if not os.environ.get("B200_GEMM_DEBUG") and not a.headline_only:  # kernel experiments produce garbage on purpose
        assert (np.diff(d_res, axis=1) <= 0).all() and (i_res >= 0).all() and (i_res < a.rows).all()
        verified = verify_results(a, index, corpus, q_host, q_dev, d_res, i_res, row0, shard_rows, N, rank, dev)

    # ---- extras beyond the headline workload (never allowed to cost the headline line)
    latency_cfg1, index_cfg3 = None, None
    if not a.headline_only:
        if rank == 0:
            try:
                latency_cfg1 = latency_extra()
            except Exception as e:
                latency_cfg1 = {"error": f"{type(e).__name__}: {e}"[:300]}
        if a.index_rows > 0:
            try:
                index.close()
                del corpus
                torch.cuda.empty_cache()
                index_cfg3 = index_extra(a, dev, N, rank, comm)
            except Exception as e:
                index_cfg3 = {"error": f"{type(e).__name__}: {e}"[:400]}
                if N > 1:
                    raise

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = peaks.get("bf16_tflops", 1590.0)
        peak_src = "MEASURED_PEAKS.json bf16_tflops (burst, of measured)" if peaks else "fallback 1590 TFLOP/s"
        flops_per_launch = 2.0 * nq * shard_rows * a.dim
        achieved = flops_per_launch / (kern_ms / max(kern_n, 1) * 1e-3) / 1e12 if kern_n else None
        out = {
            "metric": metric_name(a), "value": qps, "unit": "queries/s", "n_gpus": N, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": config_of(a, N), "clocks": clocks,
            "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": nq * a.dim * 4,
                    "d2h_bytes_per_step": nq * k * 12,
                    "note": "b200_corpus_search(): pinned host queries -> H2D -> kernels -> D2H results; corpus resident "
                            "(index state)"},
            "gpu_launches": int(launches), "verified": verified,
            "roofline": {"bound": "tensor", "kernel": "b200::gemm::gemm_topk_kernel (tcgen05 bf16 GEMM + fused top-k)",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel on this workload,
                         # from the committed ncu --set full capture (profiles/r01_gemm_topk_cg2_mc2.ncu-rep:
                         # 15.363287 GB + 8.07 MB); other shapes have no capture -> null
                         "traffic": traffic_from_profile(a, N), "traffic_unit": "bytes per launch",
                         "traffic_source": "profiles/gemm_topk_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full)",
                         "flops_per_launch": flops_per_launch, "launch_ms": kern_ms / max(kern_n, 1),
                         "launches_timed": int(kern_n), "peak_source": peak_src,
                         "hbm_algorithmic_bytes_per_launch": shard_rows * a.dim * 2},
        }
        hbm = peaks.get("hbm_gbs", 6650.0)
        for fs in flat_scan:
            if "GB_per_s" not in fs:
                continue
            fs["frac_of_hbm_peak"] = fs["GB_per_s"] / hbm
            fs["hbm_peak_GB_per_s"] = hbm
        out["flat_scan"] = flat_scan
        if fp32_batch:
            out["fp32_batch"] = fp32_batch
        if latency_cfg1:
            out["latency_cfg1"] = latency_cfg1
        if index_cfg3:
            out["index_cfg3"] = index_cfg3
        if N == 1 and not a.no_cpu_baseline and not a.headline_only:
            try:
                out["cpu_baseline"] = cpu_baseline(a)
            except Exception as e:  # never lose the GPU line to a host-side problem
                out["cpu_baseline"] = {"value": None, "unit": "queries/s", "cores": cpu_threads(), "kind": "port",
                                       "sample": f"failed: {e}"}
        print(json.dumps(out))
    if N > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
