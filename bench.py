#!/usr/bin/env python
"""bench.py — the headline measurement of the PGCN hot path on B200 (see DESIGN.md §Measurement).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W

metric  : aggregated edges/s of ONE layer's forward aggregation (PSpMM.forward = halo exchange +
          Z = A_local * H), whole job, = nnz(A^) / max-over-ranks time per step   (BASELINE.json metric)
workload: N = 1: BASELINE.json configs[1] (C2) — synthetic R-MAT 1 M vertices / 16 M edges (+ n self loops after
          the reference preprocessing), f = 128, fp32.  N > 1: configs[4] (C5) — R-MAT 10 M / 100 M, f = 128, the
          graph the north_star's scaling target is stated on, split over N ranks by the hypergraph part vector
          shipped under bench_data/ (PaToH column-net model of GPU/hypergraph/main.cpp; tools/make_partvecs.py);
          strong scaling, and rank 0 also times the SAME graph on its GPU alone (`single_gpu_same_config`) so the
          speed-up can be read from one line. `--config` overrides either default.
value   : device-resident inputs, CUDA-event timed, K steps after W warm-ups, max over ranks.
e2e     : the same step through the C-ABI host entry point pgcn_forward_host — H in pinned HOST
          memory, copied in, aggregated, Z copied back, every step.
roofline: the SpMM kernel — algorithmic bytes (SURVEY.md §8d) / CUDA-event time per launch vs the
          measured HBM copy bandwidth in MEASURED_PEAKS.json.
cpu_baseline / --impl reference: the C/OpenMP restatement of the reference's GraphBLAS aggregation
          (oracle/spmm_oracle.c, Parallel-GCN/main.c:271,295) on the host cores — the real GraphBLAS
          trainer cannot be built offline (no GraphBLAS.h / mpicc), see DESIGN.md.
--dump-outputs DIR: after the timed steps, the Z of the last step as DIR/Z.npy (float32; DIR/Z.rank<r>.npy per rank
          when N > 1) — every row when they fit in 60 MB over all ranks, else a fixed seeded sample of rows, whose
          local indices go to DIR/Z_rows.npy (float64). The inputs are seeded, so two builds run with the same
          arguments can be compared output for output.
"""
import argparse
import ctypes as C
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

METRIC = "aggregated edges/sec (SpMM) per layer"
UNIT = "edges/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=None, help="C2 | C3 | C4 | C5 (default: C2 on one GPU, C5 on several)")
    ap.add_argument("--partition", default="auto", help="auto | block | rp | path to a part vector")
    ap.add_argument("--transport", default="auto", choices=["auto", "nccl", "p2p"])
    # generated graphs are cached per user: a shared /tmp may already hold another account's unwritable cache directory
    ap.add_argument("--cache", default=os.environ.get(
        "PGCN_CACHE", os.path.join(tempfile.gettempdir(), "pgcn_b200_cache_%d" % os.getuid())))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lib-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer (e2e) measurement (side runs only)")
    ap.add_argument("--no-single", action="store_true", help="N > 1: skip the single-GPU run of the same config")
    ap.add_argument("--opt", action="append", default=[], help="plan option name=value (tuning)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step (a seeded row sample of it) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.config is None:
        args.config = "C2" if args.gpus <= 1 else "C5"
    return args


def workload_name(config):
    """One string for both arms (the driver compares them)."""
    from pgcn_b200 import graphio
    n, nnz, f, _, _ = graphio.CONFIGS[config]
    return ("%s: R-MAT %d vertices / %d edges (+%d self loops after A+I), f=%d, one forward aggregation "
            "(halo exchange + Z=A_local*H) per step" % (config, n, nnz, n, f))


def source_hash():
    """sha1 over the kernel sources: profiles/traffic_<config>.json is only quoted when it was measured on this code."""
    import hashlib
    h = hashlib.sha1()
    base = os.path.join(ROOT, "scalable-graph-convolutional-network-training-on-distributed-memory-systems_b200", "csrc")
    for name in sorted(os.listdir(base)):
        if name.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(base, name), "rb").read())
    return h.hexdigest()[:16]


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_graph(args):
    from pgcn_b200 import graphio
    return graphio.config_graph(args.config, cache_dir=args.cache)


def part_vector(args, n, k):
    from pgcn_b200 import graphio
    if k == 1:
        return np.zeros(n, dtype=np.int64), "single part"
    if args.partition not in ("auto", "block", "rp", "hp", "gp"):
        return graphio.read_partvec(args.partition, n), os.path.basename(args.partition)
    for method, what in (("hp", "hp (PaToH column-net hypergraph model of GPU/hypergraph/main.cpp, precomputed: bench_data/)"),
                         ("gp", "gp (METIS k-way of GPU/graph/main.cpp, precomputed: bench_data/)")):
        shipped = os.path.join(ROOT, "bench_data", "%s.%d.%s.npz" % (args.config, k, method))
        if args.partition in ("auto", method) and os.path.exists(shipped):
            return np.load(shipped)["partvec"].astype(np.int64), what
    if args.partition in ("hp", "gp"):
        raise SystemExit("no bench_data/%s.%d.%s.npz (tools/make_partvecs.py makes it)" % (args.config, k, args.partition))
    if args.partition == "rp":
        return graphio.random_partvec(n, k, seed=1), "rp (uniform random, seed 1)"
    return graphio.block_partvec(n, k), "block (contiguous vertex ranges)"


DUMP_BYTES = 60_000_000        # --dump-outputs: what all ranks write together stays under 64 MB


def dump_rows(m, f, world):
    """Local row indices --dump-outputs writes: all m rows when they fit the budget, else a seeded sample (sorted)."""
    cap = max(1, DUMP_BYTES // world // (4 * f + 8))
    if m <= cap:
        return np.arange(m, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(m, size=cap, replace=False))


def dump_outputs(dirname, rows, Zs, rank, world):
    """DIR/Z.npy (DIR/Z.rank<r>.npy when N > 1): Zs, the output rows `rows`, in float32; DIR/Z_rows.npy: the row
    indices (float64, exact up to 2^53)."""
    os.makedirs(dirname, exist_ok=True)
    tag = "" if world == 1 else ".rank%d" % rank
    np.save(os.path.join(dirname, "Z%s.npy" % tag), np.ascontiguousarray(Zs, dtype=np.float32))
    np.save(os.path.join(dirname, "Z_rows%s.npy" % tag), rows.astype(np.float64))


def thread_candidates(ncpu):
    """Thread counts tried for the CPU arm (the best one is reported): all logical CPUs down to 1/8 of them —
    SMT siblings and container CPU quotas often make fewer threads faster for this bandwidth/latency-bound loop."""
    return sorted({max(1, ncpu), max(1, ncpu // 2), max(1, ncpu // 4), max(1, ncpu // 8)})


def cpu_baseline(lp, f, budget_s=20.0):
    """C/OpenMP restatement of the GraphBLAS aggregation on this host's cores, same rank data."""
    from oracle import build_oracle
    rng = np.random.RandomState(1)
    H = rng.uniform(-1, 1, size=(lp.m + lp.h, f)).astype(np.float32)
    out = np.empty((lp.m, f), dtype=np.float32)
    build_oracle.spmm_csr(lp.rowptr, lp.colidx, lp.vals, H, lp.m, out=out)       # warm-up / page-in
    ncpu = os.cpu_count() or 1
    build_oracle.best_thread_count(lambda: build_oracle.spmm_csr(lp.rowptr, lp.colidx, lp.vals, H, lp.m, out=out),
                                   thread_candidates(ncpu))
    times = []
    t_all = time.perf_counter()
    while len(times) < 3 or (time.perf_counter() - t_all < budget_s and len(times) < 50):
        t0 = time.perf_counter()
        build_oracle.spmm_csr(lp.rowptr, lp.colidx, lp.vals, H, lp.m, out=out)
        times.append(time.perf_counter() - t0)
    t = float(np.median(times))
    return {"value": lp.nnz() / t, "unit": UNIT, "cores": build_oracle.num_threads(), "kind": "port",
            "sample": "full %d-edge local matrix, f=%d, median of %d passes of oracle/spmm_oracle.c (OpenMP)" % (lp.nnz(), f, len(times)),
            "ms_per_pass": t * 1e3}


def lib_baseline(A, H, n, nnz_total):
    """What the reference would do on this very GPU (SURVEY.md §8d-3), outside every timed region of the repo arm:
    torch.sparse.mm on its uncoalesced int64 COO exactly as GPU/PGCN.py:60-63,127 builds and calls it, and the same
    product on a prebuilt CSR (cuSPARSE). Library kernels — a baseline, not part of the product path."""
    import torch
    dev = H.device

    def timed(fn, iters, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    idx = torch.from_numpy(np.vstack([A.row, A.col]).astype(np.int64)).to(dev)
    val = torch.from_numpy(A.data.astype(np.float32)).to(dev)
    coo = torch.sparse_coo_tensor(idx, val, (n, n))
    ms_coo = timed(lambda: torch.sparse.mm(coo, H), 3, 1)
    csr = coo.coalesce().to_sparse_csr()
    ms_csr = timed(lambda: torch.sparse.mm(csr, H), 10, 2)
    return {"reference_call_coo": {"ms": ms_coo, "value": nnz_total / (ms_coo * 1e-3), "unit": UNIT,
                                   "what": "torch.sparse.mm on the uncoalesced int64 COO of GPU/PGCN.py:60-63,127"},
            "cusparse_csr": {"ms": ms_csr, "value": nnz_total / (ms_csr * 1e-3), "unit": UNIT,
                             "what": "torch.sparse.mm on a prebuilt CSR (cuSPARSE)"}}


def run_reference(args):
    """--impl reference: the reference's CPU aggregation (C/OpenMP restatement of the GraphBLAS path)
    on the host cores, rank 0 only, one step = one full pass over the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from pgcn_b200 import graphio, plan as planmod
    from oracle import build_oracle
    n, nnz, f, _, _ = graphio.CONFIGS[args.config]
    A = load_graph(args)
    lp = planmod.build_local_plan(A, np.zeros(n, dtype=np.int64), 0, 1)
    rng = np.random.RandomState(1)
    H = rng.uniform(-1, 1, size=(n, f)).astype(np.float32)
    out = np.empty((n, f), dtype=np.float32)
    ncpu = os.cpu_count() or 1
    build_oracle.best_thread_count(lambda: build_oracle.spmm_csr(lp.rowptr, lp.colidx, lp.vals, H, n, out=out),
                                   thread_candidates(ncpu))
    for _ in range(max(args.warmup, 1)):
        build_oracle.spmm_csr(lp.rowptr, lp.colidx, lp.vals, H, n, out=out)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        build_oracle.spmm_csr(lp.rowptr, lp.colidx, lp.vals, H, n, out=out)
    t = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        rows = dump_rows(n, f, 1)
        dump_outputs(args.dump_outputs, rows, out[rows], 0, 1)
    val = lp.nnz() / t
    cores = build_oracle.num_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "full workload per step; C/OpenMP restatement of Parallel-GCN/main.c:271,295 "
                                   "(SuiteSparse:GraphBLAS + MPI not buildable offline)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


class QuietStdout:
    """The contract is ONE JSON line on stdout: anything a library prints there while we work (NCCL's version banner
    when the box sets NCCL_DEBUG) is sent to stderr instead; `emit` writes the line to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(text, flush=True)
        os.dup2(2, 1)


def main():
    args = parse()
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # started plainly: re-launch one rank per GPU (the driver launches torch.distributed.run itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"),
               os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if args.impl == "reference":
        return run_reference(args)

    quiet = QuietStdout()
    import torch
    import torch.distributed as dist
    from pgcn_b200 import cabi, graphio, plan as planmod, op

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the PGCN B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    n, nnz, f, _, _ = graphio.CONFIGS[args.config]
    # rank 0 generates (or loads) the graph first so the cache file is written once
    if world > 1 and rank != 0:
        dist.barrier()
    A = load_graph(args)
    if world > 1 and rank == 0:
        dist.barrier()
    pv, pv_name = part_vector(args, n, world)
    lp = planmod.build_local_plan(A, pv, rank, world)
    nnz_total = int(A.nnz)
    keep_A = A if (rank == 0 and ((world > 1 and not args.no_single) or (world == 1 and not args.no_lib_baseline))) else None
    del A
    plan = planmod.PgcnPlan(lp, f, device=device)
    tuned = plan.autotune(f)          # set-up, untimed: like the reference's plan building
    for kv in args.opt:
        name, v = kv.split("=")
        plan.set_option(name, int(v))
    transport = plan.init_comm(transport=args.transport) if world > 1 else "none"

    gen = torch.Generator(device=device).manual_seed(1 + rank)
    H = torch.rand((lp.m, f), device=device, generator=gen) * 2 - 1
    Z = torch.empty((lp.m, f), device=device)
    lib = cabi.load()
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        cabi.check(lib.pgcn_forward(plan.handle, H.data_ptr(), Z.data_ptr(), f, stream), plan.handle)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- timed region: exactly K steps --------------------------------------------------------
    l0 = plan.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    sync_all()
    launches = plan.launch_count() - l0
    ms = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    # what the last timed step handed back (Z is overwritten below), untimed
    if args.dump_outputs:
        rows = dump_rows(lp.m, f, world)
        dump_outputs(args.dump_outputs, rows, Z[torch.from_numpy(rows).to(device)].cpu().numpy(), rank, world)

    # ---- the dominant kernel alone (local SpMM over [own | halo]) -----------------------------
    halo = torch.zeros((max(lp.h, 1), f), device=device)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nk = max(args.steps, 10)
    for _ in range(3):
        cabi.check(lib.pgcn_spmm(plan.handle, 0, H.data_ptr(), halo.data_ptr(), Z.data_ptr(), None, f, stream), plan.handle)
    torch.cuda.synchronize()
    k0.record()
    for _ in range(nk):
        cabi.check(lib.pgcn_spmm(plan.handle, 0, H.data_ptr(), halo.data_ptr(), Z.data_ptr(), None, f, stream), plan.handle)
    k1.record()
    torch.cuda.synchronize()
    ms_kernel = k0.elapsed_time(k1) / nk
    # backward aggregation (A^T g + reverse exchange + scatter-add), reported beside the headline
    G = torch.empty((lp.m, f), device=device)
    for _ in range(2):
        cabi.check(lib.pgcn_backward(plan.handle, Z.data_ptr(), G.data_ptr(), f, stream), plan.handle)
    sync_all()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nb = max(args.steps // 2, 5)
    b0.record()
    for _ in range(nb):
        cabi.check(lib.pgcn_backward(plan.handle, Z.data_ptr(), G.data_ptr(), f, stream), plan.handle)
    b1.record()
    sync_all()
    ms_bwd = b0.elapsed_time(b1) / nb

    # ---- e2e: host buffers through the C-ABI host entry points (software-pipelined: two device slots, the upload
    # of step i+1 and the download of step i-1 run under the aggregation of step i; every step's H goes host ->
    # device and every step's Z device -> host inside the timed region) --------------------------------------
    if args.no_e2e:
        s_e2e = s_e2e_serial = float("nan"); e2e_ok = None; n_e2e = 0
    Hh = [] if args.no_e2e else [torch.empty((lp.m, f), dtype=torch.float32).pin_memory() for _ in range(2)]
    Zh = [] if args.no_e2e else [torch.empty((lp.m, f), dtype=torch.float32).pin_memory() for _ in range(2)]
    for x in Hh:
        x.copy_(H)
    if not args.no_e2e:
        n_e2e = max(4, min(args.steps, 12))

    def e2e_run(nsteps):
        for i in range(nsteps):
            cabi.check(lib.pgcn_forward_host_async(plan.handle, Hh[i & 1].data_ptr(), Zh[i & 1].data_ptr(), f), plan.handle)
        cabi.check(lib.pgcn_forward_host_wait(plan.handle), plan.handle)

    if not args.no_e2e:
        e2e_run(2)
        sync_all()
        t0 = time.perf_counter()
        e2e_run(n_e2e)
        sync_all()
        s_e2e = (time.perf_counter() - t0) / n_e2e
        # the strictly serial form (one step at a time: copy in, aggregate, copy out, synchronise)
        t0 = time.perf_counter()
        for i in range(3):
            cabi.check(lib.pgcn_forward_host(plan.handle, Hh[0].data_ptr(), Zh[0].data_ptr(), f), plan.handle)
        sync_all()
        s_e2e_serial = (time.perf_counter() - t0) / 3
        e2e_ok = bool(torch.equal(Zh[0], Zh[1])) and bool(torch.isfinite(Zh[0][:16]).all())
    del Hh, Zh

    # ---- reduce over ranks ---------------------------------------------------------------------
    vec = torch.tensor([ms, ms_kernel, ms_bwd, s_e2e * 1e3, s_e2e_serial * 1e3, float(lp.h), float(lp.nnz())],
                       device=device, dtype=torch.float64)
    tot = torch.tensor([float(launches), float(plan.algorithmic_bytes(f)["spmm_fwd"]), float(lp.m * f * 4),
                        float(plan.algorithmic_bytes(f)["xchg_in"])], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms, ms_kernel, ms_bwd, ms_e2e, ms_e2e_serial, h_max, nnz_max = [float(x) for x in vec.tolist()]

    # ---- N > 1: the same graph on ONE GPU (rank 0 alone, the others wait), so the line carries its own baseline
    single = None
    if world > 1 and not args.no_single:
        if rank == 0:
            try:
                lp1 = planmod.build_local_plan(keep_A, np.zeros(n, dtype=np.int64), 0, 1)
                p1 = planmod.PgcnPlan(lp1, f, device=device)
                p1.autotune(f)
                H1 = torch.rand((n, f), device=device) * 2 - 1
                Z1 = torch.empty((n, f), device=device)
                for _ in range(3):
                    cabi.check(lib.pgcn_forward(p1.handle, H1.data_ptr(), Z1.data_ptr(), f, stream), p1.handle)
                torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ns = max(5, min(args.steps, 20))
                s0.record()
                for _ in range(ns):
                    cabi.check(lib.pgcn_forward(p1.handle, H1.data_ptr(), Z1.data_ptr(), f, stream), p1.handle)
                s1.record()
                torch.cuda.synchronize()
                ms1 = s0.elapsed_time(s1) / ns
                b1 = p1.algorithmic_bytes(f)["spmm_fwd"]
                single = {"ms_per_step": ms1, "value": nnz_total / (ms1 * 1e-3), "unit": UNIT, "steps": ns,
                          "roofline_frac": b1 / (ms1 * 1e-3) / 1e9 / peaks()[0]}
                p1.close()
                del H1, Z1, lp1
            except Exception as e:                      # never lose the multi-GPU number over the extra
                single = {"error": str(e)[:200]}
        dist.barrier()
    keep_A_local = keep_A
    launches_all, bytes_all, h2d_all, xchg_all = [float(x) for x in tot.tolist()]

    if rank == 0:
        peak, peak_src = peaks()
        bytes_per_rank = bytes_all / world
        achieved = bytes_per_rank / (ms_kernel * 1e-3) / 1e9
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            try:
                cpu = cpu_baseline(lp, f)
            except Exception as e:                       # the checker failing must not hide the GPU number
                cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %s" % e}
        line = {
            "metric": METRIC, "value": nnz_total / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload_name(args.config),
                "partition": pv_name, "transport": transport, "l2": "inputs larger than L2 (H and Z %.0f MB each per rank)" % (lp.m * f * 4 / 1e6),
                "plan_options": {k_: plan.get_option(k_) for k_ in ("kernel", "ring_slots", "ring_groups", "ring_edges_per_block",
                                                                    "persistent", "persistent_multi", "overlap", "relu")},
                "nnz": nnz_total, "halo_rows_rank0": int(lp.h), "send_rows_rank0": int(lp.S),
            },
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None,
                         "kernel": ("spmm_ring_g4_kernel (TMA tile::gather4 into per-warp shared-memory row rings)"
                                    if f % 128 == 0 else "spmm_rowblock_kernel (register pipeline)"),
                         "ms_per_launch": ms_kernel,
                         "algorithmic_bytes_per_launch": bytes_per_rank, "peak_source": peak_src},
            "cpu_baseline": cpu,
            "e2e": {"value": nnz_total / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_all),
                    "d2h_bytes_per_step": int(h2d_all), "ms_per_step": ms_e2e,
                    "api": "pgcn_forward_host_async + pgcn_forward_host_wait (C-ABI, pinned host buffers, two device slots: "
                           "step i+1 uploads and step i-1 downloads under the aggregation of step i)",
                    "steps": n_e2e, "serial_ms_per_step": ms_e2e_serial, "serial_api": "pgcn_forward_host", "results_equal": e2e_ok},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "backward": {"ms_per_step": ms_bwd, "value": nnz_total / (ms_bwd * 1e-3), "unit": UNIT},
            "exchange_bytes_in_per_step": int(xchg_all),
            "per_rank": {"halo_rows_max": int(h_max), "nnz_max": int(nnz_max), "spmm_alone_ms_max": ms_kernel,
                         "exchange_visible_ms": max(ms - ms_kernel, 0.0)},
        }
        if single is not None:
            line["single_gpu_same_config"] = single
            if "value" in single:
                line["speedup_vs_single_gpu"] = line["value"] / single["value"]
        if world == 1 and not args.no_lib_baseline and keep_A_local is not None:
            try:
                line["lib_baseline"] = lib_baseline(keep_A_local, H, n, nnz_total)
            except Exception as e:
                line["lib_baseline"] = {"error": str(e)[:200]}
        # DRAM bytes per launch of the dominant kernel come from an ncu capture (tools/update_traffic.py); the file is
        # stamped with the hash of the kernel sources it was measured on and ignored when the code has moved on
        traffic_file = os.path.join(ROOT, "profiles", "traffic_%s.json" % args.config)
        if os.path.exists(traffic_file) and world == 1:
            try:
                tj = json.load(open(traffic_file))
                cur = source_hash()
                if cur == tj.get("source_hash") or cur in tj.get("accepted_hashes", []):
                    line["roofline"]["traffic"] = tj.get("dram_bytes_per_launch")
                    line["roofline"]["traffic_source"] = "ncu dram__bytes_read+write per launch, %s; measured on %s%s" % (
                        tj.get("kernel", "")[:48], tj.get("measured_on_commit", "these sources")[:60],
                        "" if cur == tj.get("source_hash") else " (later sources accepted by hand, see profiles/traffic_%s.json)" % args.config)
                else:
                    line["roofline"]["traffic_source"] = "profiles/traffic_%s.json is stale (measured on other kernel sources)" % args.config
            except Exception:
                pass
        quiet.emit(json.dumps(line))
    plan.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
