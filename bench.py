#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native KNN hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA through the C ABI)
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU algorithm (oracle port)
  python bench.py ... --dump-outputs DIR                   # also save the last timed step's results as DIR/*.npy

Workload (config.workload): exact brute-force cosine KNN, k=10, batch of 1024 f64 queries per step over a
10M x 768 f32 corpus (the configuration BASELINE.json's metric is quoted on; it fits one B200).  With N
GPUs the SAME 10M-row corpus is row-sharded N ways (strong scaling); every rank screens + exactly re-ranks
its shard, ONE NCCL all-gather (issued by the library on its own stream) moves the per-shard top-k blocks and
a merge kernel on every rank produces the global top-k.  Data are synthetic: a counter-based generator
produces identical values on every GPU and on the CPU (`--data clustered`: a Gaussian mixture, see below).

Numbers on the JSON line:
  value   queries/s with the query batches resident in HBM; batches are submitted asynchronously (two in flight),
          so the device stream never waits for the host.
  e2e     queries/s through the host-buffer plugin call -- sdb_knn_bruteforce (N=1) / sdb_knn_sharded_submit +
          sdb_knn_sharded_wait (N>1) -- one synchronous call per step with pinned HOST queries and HOST results
          (H2D and D2H inside the timed region).  `e2e_pipelined` = the same buffers, two calls in flight.
  parity_checked  after the timed region the last batch is re-checked: >= 8 queries through the exact kernel
          (SDB_SCREEN_NONE_EXACT) and, at N=1, >= 2 queries through the CPU oracle over ALL rows (read back from
          the device-resident master copy); any difference in rows, order or f64 bits aborts the run.
One JSON line is printed by rank 0 (see README / the driver contract for the keys).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (rows, dim, batch, k)
    "northstar_10Mx768_b1024_k10_cosine_bruteforce": (10_000_000, 768, 1024, 10),
    "c2_1Mx768_b1024_k10_cosine_bruteforce": (1_000_000, 768, 1024, 10),
    "tiny_100kx128_b64_k10_cosine_bruteforce": (100_000, 128, 64, 10),
    # BASELINE config 4 (quoted there on 8 GPUs; 107 GB of corpus + screen copies still fit one B200)
    "c4_10Mx1536_b4096_k100_cosine_bruteforce": (10_000_000, 1536, 4096, 100),
}
SEED_CORPUS = 0x5DB00002
SEED_QUERY = 0x5DB0A000
N_CLUSTERS, CLUSTER_SIGMA = 4096, 0.15  # SURVEY C3 mixture (--data clustered)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d["bf16_tflops_sustained"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def host_threads():
    """threads this process may really use: affinity mask, capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt[0] != "max":
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota)))
    return n, quota


class ClockSampler:
    """samples SM clock and clock-event (throttle) reasons while the timed region runs.  In-process NVML from a
    thread (a ~20 us query every 5 ms); a polling `nvidia-smi -lms` child costs the GPU driver milliseconds per sample
    and visibly perturbs steps that last only a millisecond -- it is only the fallback when NVML is not importable."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self.stop_flag = index, [], None, None, False
        self.sm, self.reason_bits, self.sm_max = [], 0, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it lists plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = self.index
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                ids = [int(x) for x in vis.split(",")]
                if self.index < len(ids):
                    phys = ids[self.index]
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.reason_bits |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.t.join(timeout=1)
            n = self.nvml
            names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap),
                     ("hw_power_brake", n.nvmlClocksEventReasonHwPowerBrakeSlowdown))
            reasons = [nm for nm, bit in names if self.reason_bits & bit]
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max, "reasons": reasons,
                    "samples": len(self.sm), "source": "nvml (in-process, 5 ms period)"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5),
                          ("sw_power_cap", 6)):
            if any(len(r) >= 7 and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvidia-smi -lms 50"}


def cpu_sample(rows_total, dim, threads):
    """bounded sample of the workload for the CPU arm: the first 262144 rows, and as many queries (a multiple
    of the thread count) as fit the time budget"""
    from surrealdb_b200.synthetic import gen_f32
    sample_rows = int(min(rows_total, 262_144))
    corpus = np.empty((sample_rows, dim), np.float32)
    step = 1 << 16
    for r0 in range(0, sample_rows, step):
        r1 = min(sample_rows, r0 + step)
        corpus[r0:r1] = gen_f32(SEED_CORPUS, r0 * dim, (r1 - r0) * dim).reshape(r1 - r0, dim)
    queries = gen_f32(SEED_QUERY, 0, 64 * threads * dim).reshape(64 * threads, dim).astype(np.float64)
    return corpus, queries


def cpu_baseline(rows_total, dim, k, budget_s=12.0, threads=None, sample=None, repeats=3):
    """The ONE place bench.py touches oracle/ for timing (CPU baseline / reference arm).  Times the oracle -- a
    faithful port of the reference's f64 Vec<Number> distance + KnnTopK selection -- on the host cores this process
    may use (affinity mask and cgroup quota, not os.cpu_count()), on a bounded sample, `repeats` times; per-query
    cost is linear in rows, so the figure is scaled by sample_rows / rows_total."""
    from oracle import pyoracle as O
    hw, quota = host_threads()
    threads = threads or hw
    corpus, queries = sample if sample is not None else cpu_sample(rows_total, dim, threads)
    sample_rows = corpus.shape[0]
    t0 = time.perf_counter()  # calibration: one query per thread tells how many rounds fit the budget
    O.knn_topk_batch(corpus, queries[:threads], "cosine", k, threads)
    t_cal = time.perf_counter() - t0
    rounds = int(max(1, min(64, (budget_s / repeats) // max(t_cal, 1e-3))))
    nq = rounds * threads
    queries = queries[:nq]
    vals, dts = [], []
    for _ in range(repeats):
        t0 = time.perf_counter()
        O.knn_topk_batch(corpus, queries, "cosine", k, threads)
        dt = time.perf_counter() - t0
        dts.append(dt)
        vals.append(nq / dt * (sample_rows / rows_total))
    qps = float(np.median(vals))
    return {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
            "cores_note": f"sched_getaffinity={hw}, cgroup quota={quota}, os.cpu_count()={os.cpu_count()}",
            "repeats": repeats, "min": float(min(vals)), "max": float(max(vals)),
            "spread": float((max(vals) - min(vals)) / qps) if qps else None,
            "sample": f"{nq} queries x first {sample_rows} of {rows_total} rows, {repeats} repeats of "
                      f"{np.median(dts):.2f}s on {threads} threads (median reported), scaled by rows "
                      f"({sample_rows}/{rows_total}); the port omits the reference's KV scan + "
                      "document decode, so it is an optimistic stand-in for the Rust path"}, float(np.sum(dts))


def run_reference(args, rows, dim, batch, k, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
    threads, _ = host_threads()
    sample = cpu_sample(rows, dim, threads)
    vals, last = [], None
    t_all0 = time.perf_counter()
    for i in range(args.warmup + args.steps):
        cb, dt = cpu_baseline(rows, dim, k, budget_s=4.0, threads=threads, sample=sample, repeats=1)
        if i >= args.warmup:
            vals.append(cb["value"])
            last = cb
    qps = float(np.mean(vals))
    last["value"] = qps
    last["min"], last["max"] = float(min(vals)), float(max(vals))
    last["spread"] = float((max(vals) - min(vals)) / qps) if qps else None
    last["repeats"] = len(vals)
    out = {"impl": "reference", "metric": "KNN queries/sec @recall@10=1.0 (exact brute force)", "value": qps,
           "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": batch / qps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic", "config": {"workload": wl, "rows": rows, "dim": dim, "batch": batch,
                                                            "k": k, "metric": "cosine"},
           "cpu_baseline": last, "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0,
                                         "d2h_bytes_per_step": 0},
           "wall_s": time.perf_counter() - t_all0}
    print(json.dumps(out), flush=True)


def measure_int8_peak(torch, dev, seconds=1.5):
    """cuBLASLt int8 GEMM (torch._int_mm, s8 x s8 -> s32) 8192^3 on this GPU: burst (best of 10) and sustained
    (back to back for `seconds`) TOP/s -- the denominator of the int8 screen's roofline"""
    try:
        n = 8192
        a = torch.randint(-127, 127, (n, n), dtype=torch.int8, device=dev)
        b = torch.randint(-127, 127, (n, n), dtype=torch.int8, device=dev)
        for _ in range(3):
            torch._int_mm(a, b)
        torch.cuda.synchronize()
        ops = 2.0 * n ** 3
        best = 0.0
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            e1.synchronize()
            best = max(best, ops / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        reps = max(10, int(seconds / (ops / (best * 1e12))))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch._int_mm(a, b)
        e1.record()
        e1.synchronize()
        sustained = ops * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12
        del a, b
        return {"int8_tops": best, "int8_tops_sustained": sustained,
                "how": f"torch._int_mm (cuBLASLt s8 x s8 -> s32) {n}^3: best of 10 and {reps} back to back"}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="northstar_10Mx768_b1024_k10_cosine_bruteforce", choices=list(WORKLOADS))
    ap.add_argument("--data", default="uniform", choices=["uniform", "clustered"])
    ap.add_argument("--screen", default="AUTO")
    ap.add_argument("--schedule", default="streaming", choices=["streaming", "multipass"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the HBM-regime table and the int8 peak")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (device-resident path) to DIR as float64 .npy files: "
                         "knn_rows (global row ids), knn_dist, knn_count; the inputs depend only on the arguments, so "
                         "two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    rows, dim, batch, k = WORKLOADS[args.workload]
    if args.warmup < 3:
        args.warmup = 3 if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args, rows, dim, batch, k, args.workload)

    import torch
    import torch.distributed as dist
    from surrealdb_b200 import Context, VectorColumn
    from surrealdb_b200.sharding import shard_range
    from surrealdb_b200.synthetic import gen_f32

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ctx = Context(local)
    # Watchdog: a multi-rank run whose ranks fall out of step must END (non-zero exit), not sit in a collective until
    # somebody's time limit kills the box.  The main thread bumps `progress` at every step; 300 s without a bump = abort.
    import threading
    progress = [time.monotonic(), "start"]

    def tick(what):
        progress[0] = time.monotonic()
        progress[1] = what

    def watchdog():
        while True:
            time.sleep(5.0)
            if time.monotonic() - progress[0] > 300.0:
                sys.stderr.write(f"bench.py rank {rank}: no progress for 300 s in phase '{progress[1]}' -- aborting\n")
                sys.stderr.flush()
                os._exit(3)

    threading.Thread(target=watchdog, daemon=True).start()
    if world > 1:
        # stdout carries exactly ONE JSON line: NCCL_DEBUG=VERSION would print a banner there at communicator creation
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # the version banner / warnings must not land on stdout
        dist.init_process_group("nccl", device_id=dev)
        # the library owns its NCCL communicator: rank 0's unique id travels over the launcher's process group
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(Context.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        ctx.comm_init_rank(world, rank, bytes(uid.cpu().numpy().tobytes()))

    tick("corpus")
    # ---- shard the corpus row-wise (contiguous blocks, tile aligned); global row id = base + local ----
    base, n_local = shard_range(rows, world, rank)
    col = VectorColumn(ctx, dim, "COSINE", "F32", capacity=max(n_local, 1))
    chunk = 1 << 20
    n_batches = args.warmup + args.steps
    if args.data == "uniform":
        for r0 in range(0, n_local, chunk):
            col.append_synthetic(SEED_CORPUS, base + r0, min(chunk, n_local - r0))
        q_np = [gen_f32(SEED_QUERY + b, 0, batch * dim).reshape(batch, dim).astype(np.float64) for b in range(n_batches)]
    else:
        # SURVEY C3 mixture: 4096 Gaussian centroids on the unit sphere, noise of total norm 0.15; every 1,000,003rd
        # row carries one component blown up 50x (outlier rows).  Generated on the GPU per global 1M-row chunk, so
        # every sharding sees the same corpus.
        g = torch.Generator(device=dev)
        g.manual_seed(SEED_CORPUS)
        cent = torch.randn((N_CLUSTERS, dim), generator=g, device=dev)
        cent /= cent.norm(dim=1, keepdim=True)
        first_chunk, last_chunk = base // chunk, (base + n_local - 1) // chunk
        for ci in range(first_chunk, last_chunk + 1):
            g.manual_seed(SEED_CORPUS + 1 + ci)
            lab = torch.randint(0, N_CLUSTERS, (chunk,), generator=g, device=dev)
            x = cent[lab] + torch.randn((chunk, dim), generator=g, device=dev) * (CLUSTER_SIGMA / dim ** 0.5)
            gr = torch.arange(ci * chunk, (ci + 1) * chunk, device=dev)
            out_rows = (gr % 1_000_003) == 17
            x[out_rows, 5] *= 50.0
            lo, hi = max(base, ci * chunk), min(base + n_local, (ci + 1) * chunk)
            part = x[lo - ci * chunk: hi - ci * chunk].contiguous()
            torch.cuda.synchronize()
            col.append_device(part.data_ptr(), hi - lo)
            del x, part
        g.manual_seed(SEED_QUERY)
        q_np = []
        for b in range(n_batches):
            lab = torch.randint(0, N_CLUSTERS, (batch,), generator=g, device=dev)
            q = cent[lab] + torch.randn((batch, dim), generator=g, device=dev) * (CLUSTER_SIGMA / dim ** 0.5)
            q_np.append(q.double().cpu().numpy())
        del cent
    col.finalize()
    col.set_screen(args.screen)
    col.set_schedule(args.schedule == "streaming")
    col.set_row_base(base)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=dev)

    tick("queries")
    # ---- query batches: pinned host copies (e2e) and device-resident copies (value) ----
    q_host = [torch.from_numpy(q).pin_memory() for q in q_np]
    q_dev = [q.to(dev) for q in q_host]
    DEPTH = 2  # batches in flight
    d_out = [(torch.zeros((batch, k), dtype=torch.int64, device=dev), torch.zeros((batch, k), dtype=torch.float64, device=dev),
              torch.zeros((batch,), dtype=torch.int32, device=dev)) for _ in range(DEPTH)]
    h_out = [(torch.zeros((batch, k), dtype=torch.int64).pin_memory(), torch.zeros((batch, k), dtype=torch.float64).pin_memory(),
              torch.zeros((batch,), dtype=torch.int32).pin_memory()) for _ in range(DEPTH)]
    torch.cuda.synchronize()

    def submit_dev(b, slot):
        o = d_out[slot]
        if world > 1:
            return col.sharded_submit_device(q_dev[b].data_ptr(), batch, k, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr())
        return col.submit_device(q_dev[b].data_ptr(), batch, k, base, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr())

    def submit_host(b, slot):
        o = h_out[slot]
        if world > 1:
            return col.sharded_submit_host(q_host[b].data_ptr(), batch, k, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr())
        return col.submit_host(q_host[b].data_ptr(), batch, k, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr())

    def wait(t):
        if world > 1:
            col.sharded_wait(t)
        else:
            col.wait(t)

    screen_ms, total_ms, cand_max, reranked, survivors = [], [], [], [], []
    fallbacks = [0]

    def note_stats():
        s = col.stats()
        screen_ms.append(s["screen_ms"])
        total_ms.append(s["total_ms"])
        cand_max.append(s["n_candidates"])
        reranked.append(s["n_reranked"])
        survivors.append(s["n_survivors"])
        fallbacks[0] += s["n_fallback"]

    def run_pipelined(submit, first, last, collect):
        pending = []
        for b in range(first, last):
            tick(f"pipelined batch {b}")
            pending.append(submit(b, b % DEPTH))
            if len(pending) == DEPTH:
                wait(pending.pop(0))
                if collect:
                    note_stats()
        while pending:
            wait(pending.pop(0))
            if collect:
                note_stats()

    def run_sync_calls(first, last):
        # one synchronous plugin call per step: sdb_knn_bruteforce (host buffers) / sharded submit + wait
        o = h_out[0]
        for b in range(first, last):
            tick(f"synchronous call {b}")
            if world > 1:
                wait(submit_host(b, 0))
            else:
                import ctypes as C
                from surrealdb_b200 import _lib as L
                L.check(L.lib().sdb_knn_bruteforce(col.h, C.c_void_p(q_host[b].data_ptr()), batch, k,
                                                   C.c_void_p(o[0].data_ptr()), C.c_void_p(o[1].data_ptr()),
                                                   C.c_void_p(o[2].data_ptr()), None))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        sync_all()
        wall = (time.perf_counter() - t0) * 1e3
        ms = max(e0.elapsed_time(e1), 0.0)
        t = torch.tensor([ms, wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    tick("warm-up")
    # ---- warm-up (both paths) ----
    run_pipelined(submit_dev, 0, args.warmup, False)
    run_sync_calls(0, min(2, args.warmup))
    run_pipelined(submit_host, 0, min(4, args.warmup), False)  # (allocates the per-slot staging buffers of the host path)
    tick("timed value")
    # ---- timed: device-resident inputs (`value`) ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.kernel_launches()
    ms_value, wall_value = timed(lambda: run_pipelined(submit_dev, args.warmup, n_batches, True))
    launches = ctx.kernel_launches() - launches0
    stats = col.stats()
    if args.dump_outputs and rank == 0:
        # the slot of the last timed batch; nothing reuses d_out before the HBM-regime extras below
        o = d_out[(n_batches - 1) % DEPTH]
        os.makedirs(args.dump_outputs, exist_ok=True)
        # float64 holds every row id (< 2^53) and count exactly
        for name, t in (("knn_rows", o[0]), ("knn_dist", o[1]), ("knn_count", o[2])):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy().astype(np.float64))
    tick("timed e2e")
    # ---- timed: end to end through the host-buffer plugin call (`e2e`) ----
    ms_e2e, wall_e2e = timed(lambda: run_sync_calls(args.warmup, n_batches))
    e2e_last = (h_out[0][0].numpy().copy(), h_out[0][1].numpy().copy(), h_out[0][2].numpy().copy())
    ms_e2e_pipe, wall_e2e_pipe = timed(lambda: run_pipelined(submit_host, args.warmup, n_batches, False))
    clocks = sampler.stop() if rank == 0 else None

    tick("parity")
    # ---- parity of the last timed batch (results of the e2e pass, rows/dist on the host) ----
    parity = {"checked": 0}
    if not args.no_parity:
        last = n_batches - 1
        got_rows, got_dist, got_cnt = e2e_last
        assert (got_cnt == k).all()
        n_exact = 8
        sel = np.linspace(0, batch - 1, n_exact).astype(np.int64)
        col.set_screen("NONE_EXACT")  # the exact kernel: sequential f64 over every row, no screen
        qx = torch.from_numpy(q_np[last][sel]).pin_memory()
        xr = torch.zeros((n_exact, k), dtype=torch.int64).pin_memory()
        xd = torch.zeros((n_exact, k), dtype=torch.float64).pin_memory()
        xc = torch.zeros((n_exact,), dtype=torch.int32).pin_memory()
        if world > 1:
            wait(col.sharded_submit_host(qx.data_ptr(), n_exact, k, xr.data_ptr(), xd.data_ptr(), xc.data_ptr()))
        else:
            wait(col.submit_host(qx.data_ptr(), n_exact, k, xr.data_ptr(), xd.data_ptr(), xc.data_ptr()))
        col.set_screen(args.screen)
        ok_exact = bool((xr.numpy() == got_rows[sel]).all() and xd.numpy().tobytes() == got_dist[sel].tobytes())
        parity.update({"exact_kernel_queries": int(n_exact), "exact_kernel_equal": ok_exact})
        n_oracle = 0
        ok_oracle = True
        if world == 1 and rank == 0:
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
            from concurrent.futures import ThreadPoolExecutor
            from oracle import pyoracle as O
            osel = np.array([0, batch - 1])
            oq = q_np[last][osel]
            threads, _ = host_threads()
            step = 1 << 16
            t0 = time.perf_counter()

            def one(r0):
                n = min(step, rows - r0)
                blk = col.read_rows(r0, n)
                r, d = O.knn_topk_batch(blk, oq, "cosine", min(k, n), 1)
                return r0, r, d, blk[:2].copy() if r0 in (0, step * 7) else None

            with ThreadPoolExecutor(max_workers=max(1, min(threads, 64))) as ex:
                parts = list(ex.map(one, range(0, rows, step)))
            for qi in range(len(osel)):
                cand = []
                for r0, r, d, _ in parts:
                    cand += [(float(d[qi, j]), int(r0 + r[qi, j])) for j in range(r.shape[1])]
                # Number::cmp on floats = total order with -0 == 0; the workload has no NaN / zero rows, so (d, row) suffices
                cand.sort()
                want_rows = np.array([c[1] for c in cand[:k]], np.int64)
                want_dist = np.array([c[0] for c in cand[:k]], np.float64)
                if not ((want_rows == got_rows[osel[qi]]).all() and want_dist.tobytes() == got_dist[osel[qi]].tobytes()):
                    ok_oracle = False
            n_oracle = len(osel)
            gen_ok = True
            if args.data == "uniform":  # the device-resident bytes are the CPU generator's bytes
                for r0, _, _, head in parts:
                    if head is not None:
                        gen_ok = gen_ok and head.tobytes() == gen_f32(SEED_CORPUS, r0 * dim, 2 * dim).tobytes()
            parity.update({"oracle_queries": n_oracle, "oracle_rows": rows, "oracle_equal": ok_oracle,
                           "device_rows_equal_cpu_generator": gen_ok, "oracle_seconds": time.perf_counter() - t0})
            ok_oracle = ok_oracle and gen_ok
        parity["checked"] = int(n_exact + n_oracle)
        if not (ok_exact and ok_oracle):
            print(json.dumps({"error": "parity check failed", "parity": parity}), flush=True)
            sys.exit(3)

    tick("extras")
    # ---- HBM-bound regime (small batches), reported next to the headline: f32 streaming kernel and tensor-core screens ----
    hbm_regime = []
    int8_peak = None
    if world == 1 and not args.no_extras:
        o = d_out[0]
        for scr, b in (("SIMT_F32", 1), ("SIMT_F32", 8), ("TC_BF16", 16), ("TC_INT8", 16)):
            col.set_screen(scr)
            qd = q_dev[0][:b].contiguous()
            torch.cuda.synchronize()
            best = None
            for _ in range(4):
                col.knn_device(qd.data_ptr(), b, k, base, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr())
                s = col.stats()
                best = s if best is None or s["screen_ms"] < best["screen_ms"] else best
            byts = n_local * (dim * {"SIMT_F32": 4.0, "TC_BF16": 2.0, "TC_INT8": 1.0}[scr] + 4.0) + b * dim * 4.0
            hbm_regime.append({"screen": scr, "batch": b, "screen_ms": best["screen_ms"], "total_ms": best["total_ms"],
                               "algorithmic_bytes": byts, "GBps": byts / (best["screen_ms"] * 1e-3) / 1e9,
                               "qps": b / (best["total_ms"] * 1e-3)})
        col.set_screen(args.screen)
        int8_peak = measure_int8_peak(torch, dev)

    if rank == 0:
        pk = peaks()
        qps = batch * args.steps / (ms_value * 1e-3)
        qps_e2e = batch * args.steps / (ms_e2e * 1e-3)
        qps_e2e_pipe = batch * args.steps / (ms_e2e_pipe * 1e-3)
        scr_ms = float(np.mean(screen_ms))
        n_shard = n_local
        screen_name = {1: "SIMT_F32", 2: "TC_BF16", 3: "NONE_EXACT", 4: "TC_INT8"}.get(stats["screen_used"], "?")
        if stats["screen_used"] in (2, 4):
            flops = 2.0 * batch * n_shard * dim
            ach = flops / (scr_ms * 1e-3) / 1e12
            i8 = stats["screen_used"] == 4
            if i8 and int8_peak and "int8_tops_sustained" in int8_peak:
                peak = int8_peak["int8_tops_sustained"]
                peak_src = ("measured in this run: sustained cuBLASLt int8 GEMM (torch._int_mm 8192^3), "
                            f"burst {int8_peak['int8_tops']:.0f} TOP/s")
            elif i8:
                peak = pk["bf16_tflops_sustained"] * 2.0
                peak_src = pk["source"] + " (2 x sustained cuBLAS bf16; int8 GEMM peak not measured in this run)"
            else:
                peak = pk["bf16_tflops_sustained"]
                peak_src = pk["source"] + " (sustained cuBLAS bf16)"
            roof = {"bound": "tensor", "kernel": "screen_tc_kernel<cosine,int8> (tcgen05 kind::i8)" if i8 else "screen_tc_kernel (tcgen05 kind::f16 bf16)",
                    "achieved": ach, "peak": peak, "unit": "TOP/s" if i8 else "TFLOP/s", "frac": ach / peak,
                    "peak_source": peak_src, "traffic": None, "algorithmic_flops_per_launch": flops,
                    "launch_note": f"the screen runs as {stats['n_passes']} launch(es) of this kernel per step (a scored sample, then one streaming "
                                   "launch with in-kernel threshold refinement); 'achieved' = flops of all of them / CUDA-event time of the whole "
                                   "screen phase on the library stream (includes the selection kernels)"}
            try:  # DRAM traffic of the dominant launch, from the committed ncu capture (not re-measured here)
                tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["screen_tc_int8" if i8 else "screen_tc_bf16"]
                if rows == 10_000_000 and world == 1:
                    roof["traffic"] = tr["bytes"]
                    roof["traffic_note"] = ("dram read+write bytes of ONE launch, ncu --set full: " + tr.get("launch", "largest pass launch")
                                            + "; " + tr["source"] + f"; algorithmic bytes of that launch {tr['algorithmic_bytes_same_launch']:.4g}")
            except Exception:
                pass
        else:
            passes_over_corpus = (batch + 7) // 8
            byts = passes_over_corpus * (n_shard * dim * 4.0 + n_shard * 4.0) + batch * dim * 4.0
            ach = byts / (scr_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "screen_simt_kernel (f32 stream, 8 queries per corpus pass)",
                    "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                    "peak_source": pk["source"] + " (copy bandwidth)", "traffic": None,
                    "algorithmic_bytes_per_step": byts}
        out = {"metric": "KNN queries/sec @recall@10=1.0 (exact brute force)", "value": qps, "unit": "queries/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_value / args.steps,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": {4: "s8 screen + f64 exact", 2: "bf16 screen + f64 exact", 1: "f32 screen + f64 exact"}.get(stats["screen_used"], "f64"),
               "data": "synthetic" if args.data == "uniform" else "synthetic (clustered: 4096-centroid Gaussian mixture, sigma 0.15, outlier rows)",
               "config": {"workload": args.workload, "rows": rows, "dim": dim, "batch": batch, "k": k,
                          "metric": "cosine", "corpus_dtype": "f32 master + bf16 and int8 screen copies",
                          "screen": screen_name, "schedule": args.schedule, "exact_rerank": "f64 sequential (reference arithmetic)",
                          "sharding": f"rows/{world}", "l2": "corpus shard (>= 0.9 GB of screen copy) is larger than L2; no flush needed",
                          "batches_in_flight": DEPTH, "fallback_queries_in_timed_region": int(fallbacks[0]),
                          "candidates_reranked_per_query_mean": float(np.mean(reranked)) / batch,
                          "largest_candidate_set": int(max(cand_max)) if cand_max else 0,
                          "screen_survivors_per_query_mean": float(np.mean(survivors)) / batch if survivors else 0.0},
               "e2e": {"value": qps_e2e, "unit": "queries/s", "h2d_bytes_per_step": batch * dim * 8,
                       "d2h_bytes_per_step": batch * k * 16 + batch * 4, "ms_per_step": ms_e2e / args.steps,
                       "api": "sdb_knn_bruteforce (host buffers)" if world == 1 else "sdb_knn_sharded_submit + sdb_knn_sharded_wait (host buffers)",
                       "mode": "one synchronous call per step"},
               "e2e_pipelined": {"value": qps_e2e_pipe, "unit": "queries/s", "ms_per_step": ms_e2e_pipe / args.steps,
                                 "mode": f"same host buffers, {DEPTH} asynchronous calls in flight"},
               "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "parity_checked": parity["checked"],
               "parity": parity,
               "timing": {"value_ms_events": ms_value, "value_ms_wall": wall_value, "e2e_ms_events": ms_e2e,
                          "e2e_ms_wall": wall_e2e, "e2e_pipelined_ms_events": ms_e2e_pipe,
                          "lib_total_ms_mean": float(np.mean(total_ms)), "lib_screen_ms_mean": scr_ms}}
        if int8_peak:
            out["int8_peak"] = int8_peak
        for h in hbm_regime:
            h["frac_of_measured_hbm_peak"] = h["GBps"] / pk["hbm_gbs"]
        out["hbm_bound_regime"] = hbm_regime
        if world == 1 and not args.no_cpu_baseline:
            tick("cpu baseline")
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s"])
            out["cpu_baseline"], _ = cpu_baseline(rows, dim, k)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
