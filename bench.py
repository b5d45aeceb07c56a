#!/usr/bin/env python
"""bench.py — CSR SpMV throughput (BASELINE.json metric) on B200, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1]): random CSR 10M x 10M, 50 nnz/row, fp64, row-partitioned
over the ranks (strong scaling: the matrix is fixed, each rank owns rows/N).  A "step" is one
y = A x over the whole matrix.  The matrix comes from `legate_sparse.random` (counter-based
device generator: every N sees the SAME matrix, every rank builds only its rows); the CPU arm
regenerates the identical matrix with the generator's host twin in oracle/.

One JSON line is printed by rank 0.  Keys beyond the base contract:
  roofline      HBM roofline of the SpMV launch sequence (pipe kernel + its fix-up kernel, once per
                column block: the library splits this matrix into 2 column blocks so that the
                gathered slice of x stays L2 resident); achieved = plain-CSR algorithmic bytes / time
  e2e           the same metric through the public API with HOST vectors (pinned): N=1
                csr_array.dot(x_host, out=y_host) — 2-D blocked H2D / compute / D2H pipeline; N>1
                csr_array.dot_local(x_host, out=y_block_host): every rank uploads 1/N of x, the slices
                are all-gathered over NVLink, every rank reads back its own rows of y
  cg            CG iterations/s on the 5-point Laplacian 4096^2 (the second half of the metric), wall
                clock AND CUDA-event device time per graph replay
  spgemm        A@A on R-MAT (BASELINE configs[3] at the largest scale that fits, stated)
  powerlaw      power-law CSR 8M rows, max row 10k (BASELINE configs[4]), nnz-balanced row blocks
  cpu_baseline  the oracle's OpenMP restatement of the reference CPU task (spmv_omp.cc:36-44)
                on the host cores, FULL matrix, + the GPU result checked against it on all rows
  banded        same measurement on the reference's own microbenchmark generator
                (examples/common.py:206-249, nnz_per_row=51) — x window staged by TMA
  gathered      (N>1) the variant that all-gathers y (what the public A @ x returns)
  cusparse      (N=1, informative) cuSPARSE SpMV through torch.sparse on the same arrays —
                the vendor call the reference wraps (spmv.cu:117-152); bench-only
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "legate-sparse_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "csr_spmv_fp64_gflops"
UNIT = "GFLOP/s"
SEED = 1234
DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE_ROWS = 1 << 22     # 32 MB of float64


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--nnz-per-row", type=int, default=50)
    ap.add_argument("--no-extras", action="store_true", help="skip the banded / cg / spgemm / powerlaw / cusparse / cpu legs")
    ap.add_argument("--spgemm-scale", type=int, default=0, help="R-MAT scale of the SpGEMM leg (0 = 18 at N=1, 20 at N>=4)")
    ap.add_argument("--pl-rows", type=int, default=8_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the y of the last step to DIR/y.npy (float64; a fixed sample "
                         f"of {DUMP_SAMPLE_ROWS} rows drawn with seed {SEED} when all of y exceeds "
                         f"{DUMP_MAX_BYTES >> 20} MB), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def workload_name(args):
    return f"random CSR {args.rows}x{args.rows}, {args.nnz_per_row} nnz/row, fp64 (BASELINE configs[1])"


def gen_banded_block(r0, r1, n, k, device):
    """Rows [r0,r1) of the reference's banded ones-matrix (examples/common.py:206-249)."""
    import torch

    half = k // 2
    rows = torch.arange(r0, r1, dtype=torch.int64, device=device)
    lo = torch.clamp(rows - half, min=0)
    hi = torch.clamp(rows + half, max=n - 1)
    cnt = hi - lo + 1
    indptr = torch.zeros(r1 - r0 + 1, dtype=torch.int64, device=device)
    torch.cumsum(cnt, 0, out=indptr[1:])
    nnz = int(indptr[-1].item())
    rep = torch.repeat_interleave(torch.arange(r1 - r0, device=device), cnt)
    pos = torch.arange(nnz, dtype=torch.int64, device=device) - indptr[:-1][rep]
    cols = (lo[rep] + pos).to(torch.int32)
    vals = torch.ones(nnz, dtype=torch.float64, device=device)
    return vals, cols, indptr


# ------------------------------------------------------------------ clocks sampler
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples = []
        self.proc = None
        self.index = index

    def start(self):
        if os.environ.get("B2S_BENCH_NO_CLOCKS"):   # A/B switch: does the 10 Hz nvidia-smi poll perturb a leg?
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [t.strip() for t in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ measurement helpers
def spmv_bytes(nnz, nrows, ncols, idx_bytes):
    """Algorithmic bytes of one SpMV (SURVEY §8d): every array once."""
    return nnz * (8 + idx_bytes) + (nrows + 1) * 8 + ncols * 8 + nrows * 8


def timed_steps(fn, steps, warmup, dist_mod):
    """CUDA-event timing of `steps` calls: barrier + sync on both sides, max over ranks."""
    import torch
    import torch.distributed as td

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_mod.world_size() > 1:
        td.barrier()
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for i in range(steps):
        fn()
        evs[i + 1].record()
    torch.cuda.synchronize()
    if dist_mod.world_size() > 1:
        td.barrier()
    torch.cuda.synchronize()
    per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
    total = torch.tensor([evs[0].elapsed_time(evs[steps])], dtype=torch.float64, device="cuda")
    if dist_mod.world_size() > 1:
        td.all_reduce(total, op=td.ReduceOp.MAX)
    return float(total.item()), per


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(out_dir, y):
    """Write the full result vector y as out_dir/y.npy in float64, or, when it exceeds DUMP_MAX_BYTES, its
    values at DUMP_SAMPLE_ROWS rows drawn with SEED (sorted): the same rows for every build and rank count."""
    y = np.asarray(y, dtype=np.float64)
    if y.nbytes > DUMP_MAX_BYTES:
        rows = np.sort(np.random.default_rng(SEED).choice(y.size, size=DUMP_SAMPLE_ROWS, replace=False))
        y = y[rows]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "y.npy"), y)


def known_traffic(tag):
    """dram bytes/launch from the committed ncu --set full capture (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "spmv_traffic.json")) as f:
            return json.load(f).get(tag)
    except Exception:
        return None


# ------------------------------------------------------------------ CPU side (oracle port of the reference)
def host_threads():
    """All host threads the box offers — torchrun exports OMP_NUM_THREADS=1, which must not
    decide how many cores the CPU arm uses."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_spmv_full(n, k, budget_s, warm=1, x=None):
    """The reference's OpenMP task body (spmv_omp.cc:36-44, oracle/ref_kernels.c) on the FULL bench
    matrix regenerated by the host twin of legate_sparse.random (same seed → same matrix; arrays
    first-touched by the threads that use them).  Best over {all threads, half}."""
    from oracle import oracle

    threads_all = host_threads()
    oracle.omp_set_threads(threads_all)
    t0 = time.perf_counter()
    indptr, cols, vals = oracle.random_csr(n, n, n * k, SEED)
    if x is None:
        x = oracle.fill_uniform(n, 1)
    gen_s = time.perf_counter() - t0
    best, y = None, None
    for threads in sorted({threads_all, max(1, threads_all // 2)}, reverse=True):
        oracle.omp_set_threads(threads)
        for _ in range(warm):
            y = oracle.spmv(indptr, cols, vals, x, omp=True)
        reps, t1 = 0, time.perf_counter()
        while reps < 3 or (time.perf_counter() - t1 < budget_s / 2 and reps < 200):
            y = oracle.spmv(indptr, cols, vals, x, omp=True)
            reps += 1
        dt = (time.perf_counter() - t1) / reps
        if best is None or dt < best[0]:
            best = (dt, threads, reps)
    dt, threads, reps = best
    info = {"seconds_per_spmv": dt, "threads": threads, "reps": reps, "generate_s": gen_s,
            "host_cpus": os.cpu_count(), "threads_available": threads_all}
    return info, (indptr, cols, vals, x, y)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = its OpenMP task body
    (spmv_omp.cc:36-44), restated in oracle/ref_kernels.c (the native reference cannot be built
    here: legate.h), all host threads, on the SAME matrix as the GPU arm (full size)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    k, n = args.nnz_per_row, args.rows
    info, (_, _, _, _, y) = cpu_spmv_full(n, k, budget_s=max(4.0, 0.5 * args.steps), warm=max(1, min(args.warmup, 3)))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y)
    dt = info["seconds_per_spmv"]
    gflops = 2.0 * n * k / dt / 1e9
    sample = (f"the full {n}x{n} matrix ({n * k} nnz) per step, int64 column ids, identical to the GPU arm's matrix "
              f"(host twin of legate_sparse.random, seed {SEED}); {info['reps']} timed passes")
    line = {
        "impl": "reference", "metric": METRIC, "value": gflops, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "rows": n, "nnz": n * k, "index_dtype": "int64", "sample": sample,
                   "same_matrix_as_gpu_arm": True},
        "cpu_baseline": {"value": gflops, "unit": UNIT, "cores": info["threads"], "kind": "port", "sample": sample,
                         "threads_available": info["threads_available"], "host_cpus": info["host_cpus"]},
        "e2e": {"value": gflops, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------ own arm
def plan_info_of(A):
    """tiling of the cached plan, or the column-block layout when the library chose one"""
    blk = A._block()
    if blk.colblock:
        return {"colblock": blk.colblock.info()}
    return blk.plan.info()


def run_b200(args):
    import torch

    import legate_sparse as sparse
    from legate_sparse import _native, dist

    dist.init()
    G, rank = dist.world_size(), dist.rank()
    assert G == args.gpus or (args.gpus == 1 and G == 1), f"--gpus {args.gpus} but WORLD_SIZE={G}"
    dev = torch.device("cuda", torch.cuda.current_device())
    n, k = args.rows, args.nnz_per_row
    bounds = dist.row_block_bounds(n, G)
    r0, r1 = int(bounds[rank]), int(bounds[rank + 1])

    # the public generator: this rank's rows only, same matrix for every N
    A = sparse.random(n, n, density=k / n, rng=SEED, dtype=np.float64)
    blk = A._block()
    vals, cols, indptr = blk.data, blk.indices, blk.indptr
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    x = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
    x_host = torch.empty(n, dtype=torch.float64).pin_memory()
    x_host.copy_(x)
    x_np = x_host.numpy()          # the checker legs (oracle rows, CPU baseline) multiply the same vector
    y_loc = torch.empty(r1 - r0, dtype=torch.float64, device=dev)
    t_build = time.perf_counter()
    A.dot_local(x, out=y_loc)  # builds the plan / column-blocked operand (one-time, like Legate's cached partitions)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t_build) * 1e3
    nnz_total = n * k
    plan_info = plan_info_of(A)

    # size-independent parity property at FULL size: linearity + a row sample against the oracle
    parity = full_size_checks(A, x, y_loc, vals, cols, indptr, r0)

    clocks = Clocks(torch.cuda.current_device())
    clocks.start()
    launches0 = _native.launch_count()
    total_ms, per = timed_steps(lambda: A.dot_local(x, out=y_loc), args.steps, args.warmup, dist)
    # the counter spans warm-up + timed calls (same launches per call): keep the timed share
    launches = (_native.launch_count() - launches0) * args.steps // (args.steps + args.warmup)
    if args.dump_outputs:
        y_all = dist.allgather_rows(y_loc, bounds)      # collective: every rank takes part
        if rank == 0:
            dump_outputs(args.dump_outputs, y_all.cpu().numpy())
        del y_all
    ms_per_step = total_ms / args.steps
    value = 2.0 * nnz_total / (ms_per_step * 1e-3) / 1e9

    # roofline of the local launch sequence (rank 0's block; at N=1 the whole matrix)
    nnz_loc = int(vals.numel())
    B_local = spmv_bytes(nnz_loc, r1 - r0, n, 4)
    kernel_ms = float(np.mean(per))
    peak, peak_src = peaks()
    achieved = B_local / (kernel_ms * 1e-3) / 1e9
    nbk = plan_info["colblock"]["nblocks"] if "colblock" in plan_info else 1   # pipe-kernel launches per step
    req_ceiling = None
    if nbk > 1:
        # the dominant kernel's own ceiling: one L2 request per clock per SM (l1tex→xbar port, ncu:
        # l1tex__m_l1tex2xbar_req_cycles_active 90 %): gathers + 128-byte stream requests
        reqs = nnz_loc + (nnz_loc * 12) / 128.0
        req_ceiling = {"requests_per_step": reqs, "ceiling_ms": reqs / (148 * 1.965e9) * 1e3,
                       "frac_of_ceiling": reqs / (148 * 1.965e9) * 1e3 / kernel_ms,
                       "evidence": "profiles/r2_gather_paths.txt, profiles/r2_ncu_spmv_pipe.md"}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": known_traffic(f"random_n{n}_k{k}_g{G}" + (f"_cb{nbk}" if nbk > 1 else "")),
                "launches_per_step": nbk, "algorithmic_bytes_per_launch": B_local / nbk, "idx_bytes": 4,
                "kernel_ms": kernel_ms / nbk,
                "peak_source": peak_src, "frac_of_8000_spec": achieved / 8000.0,
                "l2_request_ceiling": req_ceiling,
                "timed": "the launch sequence of one SpMV call, CUDA events per step: spmv_pipe_kernel + "
                         "spmv_fixup_kernel, once per column block when the operand is column-blocked "
                         "(achieved counts the plain-CSR algorithmic bytes once, not the extra indptr/y passes)"}

    # ---- e2e: public API with host buffers (pinned), copies inside the timed region
    if G == 1:
        y_host = torch.empty(n, dtype=torch.float64).pin_memory()

        def e2e_step():
            A.dot(x_host, out=y_host)

        d2h = n * 8
        h2d = n * 8
        path = ("csr_array.dot(x_pinned_host, out=y_pinned_host): 2-D blocked pipeline — x uploaded slice by slice "
                "while earlier column blocks run, finished row chunks of y copied back while later chunks run; "
                "matrix resident in HBM")
    else:
        y_host = torch.empty(r1 - r0, dtype=torch.float64).pin_memory()

        def e2e_step():
            A.dot_local(x_host, out=y_host)

        h2d = (n // G) * 8
        d2h = (r1 - r0) * 8
        path = ("csr_array.dot_local(x_pinned_host, out=y_block_pinned_host): every rank uploads 1/N of x, NCCL "
                "all-gather of x over NVLink, SpMV of its row block, D2H of its rows of y (y row-sharded on the hosts "
                "like the headline); bytes are per rank")
    e2e_steps = max(3, min(args.steps, 10))
    e2e_step()
    e2e_ms, _ = timed_steps(e2e_step, e2e_steps, 3, dist)
    torch.cuda.synchronize()
    # e2e parity: the host result equals the device-resident result
    e2e_err = float((y_host.to(dev) - y_loc).abs().max().item())
    e2e_val = 2.0 * nnz_total / (e2e_ms / e2e_steps * 1e-3) / 1e9
    e2e = {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": e2e_ms / e2e_steps, "max_abs_diff_vs_device_path": e2e_err, "path": path}

    colblock_cfg = None
    if "colblock" in plan_info:
        colblock_cfg = {"blocks": nbk, "extra_hbm_bytes": int(nnz_loc * 12 + nbk * (r1 - r0 + 1) * 8),
                        "what": "second copy of cols+vals split by column block + per-block indptr "
                                "(+ the same again for the host-vector pipeline's 2-D blocks, built on first use)",
                        "first_call_ms_incl_build": build_ms}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": G, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args), "rows": n, "nnz": nnz_total, "index_dtype": "int32",
                   "generator": f"legate_sparse.random(n, n, density={k}/n, rng={SEED}) — counter-based, on the device",
                   "partition": f"1-D row blocks over {G} rank(s), x replicated, y row-sharded",
                   "l2": "per-step inputs (%.2f GB/rank) exceed the 126 MB L2; no flush between steps"
                         % (B_local / 1e9),
                   "plan": plan_info, "colblock": colblock_cfg},
        "effective_hbm_gbs": G * achieved if G == 1 else None,
        "clocks": None, "e2e": e2e, "gpu_launches": int(launches) * G, "roofline": roofline, "parity": parity,
    }

    # ---- gathered-y variant (what the public A @ x returns) at N>1, checked against the oracle
    if G > 1:
        y_full = dist.replicated_empty(n, torch.float64)     # symmetric memory: the kernel stores into it directly
        g_ms, _ = timed_steps(lambda: A.dot(x, out=y_full), args.steps, args.warmup, dist)
        rows = torch.linspace(0, n - 1, 512, device=dev).long().unique()
        want = oracle_rows(rows.cpu().numpy(), n, k, x_np)
        got = y_full[rows].cpu().numpy()
        gerr = float(np.linalg.norm(got - want) / np.linalg.norm(want))
        own = float((y_full[r0:r1] - y_loc).abs().max().item())
        assert gerr < 1e-10 and own == 0.0, (gerr, own)
        line["gathered"] = {"value": 2.0 * nnz_total / (g_ms / args.steps * 1e-3) / 1e9, "unit": UNIT,
                            "ms_per_step": g_ms / args.steps, "oracle_rows_checked": int(rows.numel()),
                            "oracle_relerr": gerr,
                            "what": "A.dot(x, out=dist.replicated_empty(n)): SpMV with the all-gather of y fused into the "
                                    "kernel stores (NVLink P2P straight into every rank's copy of the caller's symmetric out "
                                    "buffer, opening + closing barrier, no staging copy; NCCL all-gather when peer memory is "
                                    "unavailable); rows from EVERY rank's block checked against the oracle"}

    if not args.no_extras:
        del A, blk
        if G > 1:
            del y_full
        torch.cuda.empty_cache()
        line["banded"] = banded_leg(args, dist, dev, bounds, rank, peak)
        line["cg"] = cg_leg(dist, dev, rank)
        line["powerlaw"] = powerlaw_leg(args, dist, dev, rank, peak)
        line["spgemm"] = spgemm_leg(args, dist, dev, rank)
        if G == 1 and rank == 0:
            line["cusparse"] = cusparse_leg(vals, cols, indptr, x, n, args)
            line["cpu_baseline"] = cpu_baseline_leg(args, y_loc, x_np)
    line["clocks"] = clocks.stop()   # sampled from the first timed region to the last one
    if rank == 0:
        print(json.dumps(line))
    dist.shutdown()


def oracle_rows(rows, n, k, x_np):
    """y[rows] of the bench matrix by the oracle: rows regenerated by the generator's host twin,
    multiplied by the reference's C loop (spmv.cc:36-43)."""
    from oracle import oracle

    out = np.empty(len(rows))
    for i, r in enumerate(rows.tolist()):
        p, c, v = oracle.random_csr(n, n, n * k, SEED, r0=r, r1=r + 1)
        out[i] = oracle.spmv(p, c, v, x_np)[0]
    return out


def full_size_checks(A, x, y_loc, vals, cols, indptr, r0):
    """Parity at full size: (i) linearity A(2x) == 2 A x to round-off, (ii) 2048 sampled rows
    recomputed by the oracle's C loop (reference spmv.cc:36-43) within 1e-10 relative."""
    import torch

    from oracle import oracle

    y2 = A.dot_local(2.0 * x)
    lin = float((torch.linalg.vector_norm(y2 - 2.0 * y_loc) / torch.linalg.vector_norm(y_loc)).item())
    nloc = y_loc.numel()
    rows = torch.linspace(0, nloc - 1, 2048, device=y_loc.device).long().unique()
    lo, hi = indptr[rows], indptr[rows + 1]
    cnt = (hi - lo)
    sub_ptr = np.concatenate([[0], np.cumsum(cnt.cpu().numpy())]).astype(np.int64)
    sel = torch.cat([torch.arange(int(a), int(b), device=rows.device) for a, b in zip(lo.tolist(), hi.tolist())])
    sub_cols = cols[sel].cpu().numpy().astype(np.int64)
    sub_vals = vals[sel].cpu().numpy()
    y_or = oracle.spmv(sub_ptr, sub_cols, sub_vals, x.cpu().numpy())
    y_gpu = y_loc[rows].cpu().numpy()
    err = float(np.linalg.norm(y_gpu - y_or) / np.linalg.norm(y_or))
    assert lin < 1e-14 and err < 1e-10, (lin, err)
    return {"linearity_relerr": lin, "oracle_rows_checked": int(rows.numel()), "oracle_relerr": err,
            "tolerance": 1e-10}


def cg_leg(dist, dev, rank, grid=4096, iters=1000):
    """BASELINE metric, second half: CG iterations/s on the 5-point Laplacian (config 3: 4096^2 grid,
    fp64), fixed iteration count (no early exit), fused kernels, all ranks.  Wall clock around the
    solver call AND CUDA-event device time per graph replay (25 iterations per replay); at N>1 the
    iterate after 50 iterations is checked against the oracle's CG on rank 0's rows."""
    import torch

    import legate_sparse as sparse
    import legate_sparse.linalg as linalg
    from side_bench import poisson2d_block

    G = dist.world_size()
    n = grid * grid
    bounds = dist.row_block_bounds(n, G)
    r0, r1 = int(bounds[rank]), int(bounds[rank + 1])
    data, idx, ptr = poisson2d_block(grid, r0, r1, dev)
    A = sparse.csr_array.from_row_block(data, idx, ptr, (n, n), row_start=r0, bounds=bounds)
    g = torch.Generator(device=dev)
    g.manual_seed(2)
    b = torch.rand(n, dtype=torch.float64, device=dev, generator=g)
    x50, _ = linalg.cg(A, b, rtol=0.0, atol=0.0, maxiter=50)
    torch.cuda.synchronize()
    check = cg_iterate_check(grid, b, x50) if rank == 0 else None

    def call(m):
        if G > 1:
            import torch.distributed as td

            td.barrier()
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, done = linalg.cg(A, b, rtol=0.0, atol=0.0, maxiter=m)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, done

    # whole solver call (set-up: graph capture, halo ranges, scalars + `iters` iterations), and the
    # steady iteration rate from the difference to a short call (the set-up is the same in both)
    dt_short, it_short = call(iters // 5)
    os.environ["LEGATE_SPARSE_CG_PROFILE"] = "1"
    dt, it = call(iters)
    os.environ["LEGATE_SPARSE_CG_PROFILE"] = "0"
    prof = linalg.cg_profile()
    dev_ms = sum(ms for (_, ms) in prof)
    dev_it = sum(k for (k, _) in prof)
    steady = (it - it_short) / max(dt - dt_short, 1e-9)
    nnz = A.nnz
    ref_bytes = nnz * 12 + (n + 1) * 8 + 16 * n + 120 * n
    fused_bytes = ref_bytes - 48 * n
    peak, _ = peaks()
    dev_rate = dev_it / (dev_ms * 1e-3) if dev_ms > 0 else None
    return {"workload": f"CG, 5-point Laplacian {grid}x{grid} (n={n}, nnz={nnz}), fp64, identity M, {it} iterations",
            "iters_per_s": it / dt, "ms_per_iter": dt / it * 1e3, "steady_iters_per_s": steady,
            "device_iters_per_s": dev_rate, "device_ms_per_iter": dev_ms / dev_it if dev_it else None,
            "device_timed_iterations": dev_it, "graph_replays": len(prof),
            "timing": "wall clock around linalg.cg() incl. its set-up; steady = (it - it/5) / (t - t_short); device = "
                      "CUDA events around every CUDA-graph replay (25 iterations per replay) on the launching stream",
            "reference_algorithm_bytes_per_iter": ref_bytes, "fused_bytes_per_iter": fused_bytes,
            "fused_frac_of_hbm_peak_device_time": (fused_bytes / G) * dev_rate / 1e9 / peak if dev_rate else None,
            "iterate_check_50_iterations": check,
            "comm": ("none (single GPU)" if G == 1 else
                     "per iteration: halo of p by NVLink P2P stores inside the p-update kernel + 3 one-warp board exchanges "
                     "(flags / p.q / r.r: in-kernel all-reduce over peer-mapped memory, no NCCL in the graph)"),
            "kernels_per_iter": "cg_pupdate(+halo) + spmv_pipe(+dot) + fixup + reduce + cg_update (+3 board exchanges at N>1)"}


def cg_iterate_check(grid, b, x50):
    """The distributed iterate after 50 fixed iterations equals the oracle's CG (numpy restatement of
    reference linalg.py:465-535, scipy matvec) on a subsampled set of entries."""
    import scipy.sparse as sp

    from oracle import oracle

    if grid > 4096:
        return None
    n = grid * grid
    main = np.full(n, 4.0)
    off1 = np.full(n - 1, -1.0)
    off1[np.arange(1, n) % grid == 0] = 0
    offn = np.full(n - grid, -1.0)
    S = sp.diags([offn, off1, main, off1, offn], [-grid, -1, 0, 1, grid], format="csr")
    xo, _ = oracle.cg(lambda v: S @ v, b.cpu().numpy(), rtol=0.0, atol=0.0, maxiter=50)
    xs = x50.cpu().numpy() if hasattr(x50, "cpu") else np.asarray(x50)
    err = float(np.linalg.norm(xs - xo) / np.linalg.norm(xo))
    assert err < 1e-10, err
    return {"relerr_vs_oracle_cg": err, "tolerance": 1e-10}


def banded_leg(args, dist, dev, bounds, rank, peak):
    import torch

    import legate_sparse as sparse

    n, k = args.rows, 51
    r0, r1 = int(bounds[rank]), int(bounds[rank + 1])
    vals, cols, indptr = gen_banded_block(r0, r1, n, k, dev)
    A = sparse.csr_array.from_row_block(vals, cols, indptr, (n, n), row_start=r0, bounds=bounds)
    x = torch.ones(n, dtype=torch.float64, device=dev)
    y = torch.empty(r1 - r0, dtype=torch.float64, device=dev)
    A.dot_local(x, out=y)
    ok = bool((y[100:-100] == 51.0).all().item()) if (r1 - r0) > 400 else True
    ms, per = timed_steps(lambda: A.dot_local(x, out=y), args.steps, args.warmup, dist)
    nnz_loc = int(vals.numel())
    t = torch.tensor([nnz_loc], dtype=torch.float64, device=dev)
    dist.allreduce_sum_(t)
    nnz_total = float(t.item())
    B = spmv_bytes(nnz_loc, r1 - r0, n, 4)
    ach = B / (float(np.mean(per)) * 1e-3) / 1e9
    return {"workload": f"banded ones {n}x{n}, 51 nnz/row (reference examples/common.py:206-249)",
            "value": 2.0 * nnz_total / (ms / args.steps * 1e-3) / 1e9, "unit": UNIT,
            "ms_per_step": ms / args.steps, "interior_rows_exact": ok,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak},
            "plan": plan_info_of(A)}


def powerlaw_matrix(n, dev):
    """BASELINE config 5: power-law row degrees P(d) ~ d^-2 clipped to [1, 10000] (one row forced to
    10000), uniform columns, seed 7 — the same generator as tools/side_bench.py powerlaw."""
    import torch

    g = torch.Generator(device=dev)
    g.manual_seed(7)
    u = torch.rand(n, device=dev, generator=g, dtype=torch.float64)
    deg = torch.clamp((1.0 / (1.0 - u * (1.0 - 1.0 / 10000.0))).floor().long(), 1, 10000)
    deg[n // 3] = 10000
    ptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    torch.cumsum(deg, 0, out=ptr[1:])
    nnz = int(ptr[-1].item())
    cols = torch.randint(0, n, (nnz,), device=dev, generator=g, dtype=torch.int32)
    vals = torch.rand(nnz, device=dev, generator=g, dtype=torch.float64) - 0.5
    x = torch.rand(n, device=dev, generator=g, dtype=torch.float64)
    return vals, cols, ptr, x, nnz


def powerlaw_leg(args, dist, dev, rank, peak):
    """SpMV on the power-law matrix, nnz-balanced row blocks (equal rows would starve ranks), y
    row-sharded; oracle check on sampled rows incl. the longest one; cuSPARSE beside it at N=1."""
    import torch

    import legate_sparse as sparse
    from oracle import oracle

    G = dist.world_size()
    n = args.pl_rows
    vals, cols, ptr, x, nnz = powerlaw_matrix(n, dev)      # every rank generates the same arrays
    bounds = dist.nnz_balanced_bounds(ptr, G)
    r0, r1 = int(bounds[rank]), int(bounds[rank + 1])
    lo, hi = int(ptr[r0].item()), int(ptr[r1].item())
    A = sparse.csr_array.from_row_block(vals[lo:hi].clone(), cols[lo:hi].clone(), (ptr[r0:r1 + 1] - lo).clone(), (n, n),
                                        row_start=r0, bounds=bounds)
    y = torch.empty(r1 - r0, dtype=torch.float64, device=dev)
    A.dot_local(x, out=y)
    # parity: sampled local rows + the longest row, the reference's C loop
    xs = x.cpu().numpy()
    rows = torch.linspace(r0, r1 - 1, 300).long().unique().tolist()
    if r0 <= n // 3 < r1:
        rows.append(n // 3)
    worst = 0.0
    for r in rows:
        a, b = int(ptr[r].item()), int(ptr[r + 1].item())
        ref = oracle.spmv(np.array([0, b - a]), cols[a:b].cpu().numpy(), vals[a:b].cpu().numpy(), xs)[0]
        worst = max(worst, abs(float(y[r - r0]) - ref) / max(abs(ref), 1e-300))
    assert worst < 1e-10, worst
    ms, per = timed_steps(lambda: A.dot_local(x, out=y), args.steps, args.warmup, dist)
    ms_step = ms / args.steps
    nnz_loc = hi - lo
    B = spmv_bytes(nnz_loc, r1 - r0, n, 4)
    ach = B / (float(np.mean(per)) * 1e-3) / 1e9
    out = {"workload": f"power-law CSR n={n}, nnz={nnz}, max row 10000, uniform columns (BASELINE configs[4])",
           "value": 2.0 * nnz / (ms_step * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms_step,
           "partition": f"nnz-balanced row blocks over {G} rank(s) (dist.nnz_balanced_bounds), y row-sharded",
           "rows_checked_vs_oracle": len(rows), "max_rel_err_vs_oracle_rows": worst, "tolerance": 1e-10,
           "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak},
           "plan": plan_info_of(A)}
    if G == 1:
        try:
            At = torch.sparse_csr_tensor(ptr.to(torch.int32), cols, vals, size=(n, n))
            for _ in range(3):
                At @ x
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                At @ x
            e1.record()
            torch.cuda.synchronize()
            cms = e0.elapsed_time(e1) / 10
            out["cusparse"] = {"ms_per_step": cms, "value": 2.0 * nnz / cms / 1e6, "unit": UNIT,
                               "what": "cusparseSpMV via torch.sparse_csr_tensor @ x, incl. y allocation"}
        except Exception as e:
            out["cusparse"] = {"unavailable": str(e)[:160]}
    return out


def spgemm_leg(args, dist, dev, rank):
    """BASELINE configs[3]: C = A @ A on R-MAT (edge factor 16, (a,b,c,d) = (.57,.19,.19,.05), seed 42).
    Scale 22 does not fit: nnz(C) grows ~8x per 2 scales (1.28 G at scale 18 ⇒ ~80 G entries ≈ 1 TB
    at scale 22) — the largest scale whose row-sharded C fits is used and stated.  A is row-blocked,
    B replicated, C stays ROW-SHARDED (only per-rank nnz is exchanged, like the reference)."""
    import torch

    import legate_sparse as sparse
    from side_bench import rmat_device

    G = dist.world_size()
    scale = args.spgemm_scale or (18 if G < 4 else 20)
    data, idx, ptr, n = rmat_device(scale, device=dev)        # same matrix on every rank
    nnzA = int(data.numel())
    A = sparse.csr_array((data, idx, ptr), shape=(n, n))
    partition = f"A row-blocked over {G} rank(s) (equal rows), B replicated"
    if G > 2:
        # R-MAT rows are skewed: equal-row blocks leave 2/3 of C on rank 0 (at scale 20 that is what has to fit).
        # Balance the intermediate products per rank instead (rows weighted by sum_k nnz(B_k)).  At 2 ranks the
        # equal-row split is kept: measured 136 ms vs 232 ms product-balanced (profiles/r2_bench_n2.json before /
        # after) — the heavy rows of the dense-accumulator class, not the products, set the time there.
        row_nnzB = (ptr[1:] - ptr[:-1]).to(torch.float64)
        w = torch.zeros(n, dtype=torch.float64, device=dev)
        rows = torch.repeat_interleave(torch.arange(n, device=dev), (ptr[1:] - ptr[:-1]))
        w.index_add_(0, rows, row_nnzB[idx.long()])
        A.set_row_bounds(dist.weight_balanced_bounds(w, G))
        partition = f"A row-blocked over {G} rank(s), rows weighted by their intermediate products, B replicated"
        del w, rows, row_nnzB
    try:
        C = A @ A   # warm-up (allocations)
        C = None
        torch.cuda.synchronize()
        reps = 3
        if G > 1:
            import torch.distributed as td

            td.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            C = None          # release the previous product first: C is 15 GB at scale 18
            C = A @ A
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        if G > 1:
            import torch.distributed as td

            td.all_reduce(ms, op=td.ReduceOp.MAX)
        ms = float(ms.item())
        prod = C._last_products
        nnzC = C.nnz
        blk = C._block()
        # parity at this size: sampled local rows against the oracle's Gustavson (reference
        # spgemm_csr_csr_csr.cc:62-87,134-158), sorted by column
        check = spgemm_row_check(data, idx, ptr, n, blk)
        low = ((2 * nnzA + nnzC) * 12 + 3 * (n + 1) * 8)
        out = {"workload": f"R-MAT scale {scale} (n={n}, nnz(A)={nnzA}): C = A @ A, fp64, int32 column ids",
               "scale": scale, "why_not_scale_22": "nnz(C) ~ 80 G entries (~1 TB) exceeds 8 x 180 GB; largest fitting scale used",
               "ms": ms, "products": prod, "products_per_s": prod / (ms * 1e-3), "gflops": 2.0 * prod / ms / 1e6,
               "nnzC": nnzC, "compression": prod / max(nnzC, 1),
               "lower_bound_bytes": low, "lower_bound_gbs": low / ms / 1e6,
               "partition": partition + ", C row-sharded (per-rank nnz all-gathered only)",
               "local_nnzC": blk.nnz, "rows_checked_vs_oracle": check}
        if G == 1:
            try:
                At = torch.sparse_csr_tensor(ptr, idx.long(), data, size=(n, n))
                Ct = torch.sparse.mm(At, At)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                Ct = torch.sparse.mm(At, At)
                torch.cuda.synchronize()
                out["cusparse_ms"] = (time.perf_counter() - t0) * 1e3
                out["cusparse_nnzC"] = int(Ct._nnz())
                del At, Ct
            except Exception as e:
                out["cusparse_error"] = str(e)[:160]
        del C
    except RuntimeError as e:
        out = {"workload": f"R-MAT scale {scale}", "error": str(e)[:300]}
    del A
    torch.cuda.empty_cache()
    return out


def spgemm_row_check(data, idx, ptr, n, blkC, nrows=24):
    from oracle import oracle
    import torch

    ip, ix, dv = ptr.cpu().numpy(), idx.cpu().numpy().astype(np.int64), data.cpu().numpy()
    rows = torch.linspace(blkC.r0, blkC.r1 - 1, nrows).long().unique().tolist()
    cptr = blkC.indptr
    worst = 0.0
    for r in rows:
        a_ptr = np.array([0, ip[r + 1] - ip[r]], dtype=np.int64)
        cp, ci, cv = oracle.spgemm(a_ptr, ix[ip[r]:ip[r + 1]], dv[ip[r]:ip[r + 1]], ip, ix, dv, n)
        order = np.argsort(ci, kind="stable")
        lo, hi = int(cptr[r - blkC.r0].item()), int(cptr[r - blkC.r0 + 1].item())
        gi = blkC.indices[lo:hi].cpu().numpy().astype(np.int64)
        gv = blkC.data[lo:hi].cpu().numpy()
        assert np.array_equal(gi, ci[order]), r
        worst = max(worst, float(np.max(np.abs(gv - cv[order]) / np.maximum(np.abs(cv[order]), 1e-300))) if len(gv) else 0.0)
    assert worst < 1e-10, worst
    return {"rows": len(rows), "structure_exact": True, "max_rel_err": worst, "tolerance": 1e-10}


def cusparse_leg(vals, cols, indptr, x, n, args):
    """Vendor baseline (bench-only, never linked into the product): torch.sparse CSR @ x → cusparseSpMV."""
    import torch

    try:
        At = torch.sparse_csr_tensor(indptr.to(torch.int32), cols, vals, size=(n, n))
        for _ in range(3):
            yt = At @ x
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = max(3, min(args.steps, 10))
        e0.record()
        for _ in range(steps):
            yt = At @ x
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        del yt
        return {"value": 2.0 * vals.numel() / (ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms,
                "what": "cusparseSpMV via torch.sparse_csr_tensor @ x (int32 indices), includes y allocation"}
    except Exception as e:  # informative leg only
        return {"unavailable": str(e)[:200]}


def cpu_baseline_leg(args, y_gpu, x_np):
    """Oracle port of the reference's OpenMP task on the host cores, FULL matrix (about 10-20 s incl.
    generating it), and the GPU's y checked against the CPU's y on ALL rows."""
    import scipy.sparse as sp

    k, n = args.nnz_per_row, args.rows
    info, (indptr, cols, vals, x, y_cpu) = cpu_spmv_full(n, k, budget_s=8.0, x=np.ascontiguousarray(x_np))
    dt = info["seconds_per_spmv"]
    yg = y_gpu.cpu().numpy()
    err = float(np.linalg.norm(yg - y_cpu) / np.linalg.norm(y_cpu))
    assert err < 1e-10, err
    rows_s = min(n, 1_000_000)
    S = sp.csr_array((vals[: rows_s * k], cols[: rows_s * k].astype(np.int32), indptr[: rows_s + 1].astype(np.int32)),
                     shape=(rows_s, n))
    S @ x
    t1 = time.perf_counter()
    for _ in range(3):
        S @ x
    dts = (time.perf_counter() - t1) / 3
    return {"value": 2.0 * n * k / dt / 1e9, "unit": UNIT, "cores": info["threads"], "kind": "port",
            "sample": f"the full {n}x{n} matrix ({n * k} nnz), {info['reps']} passes of the OpenMP SpMV "
                      f"(oracle restatement of spmv_omp.cc:36-44), matrix regenerated on the host in {info['generate_s']:.1f} s",
            "full_y_relerr_gpu_vs_cpu": err, "rows_compared": n, "tolerance": 1e-10,
            "scipy_single_thread_gflops": 2.0 * rows_s * k / dts / 1e9,
            "host_cpus": info["host_cpus"], "threads_available": info["threads_available"]}


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
