#!/usr/bin/env python
"""bench.py — FCMA correlation hot path: voxel-pair correlations / second.

  python bench.py --gpus N --steps K --warmup W            # B200 arm (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference's own CPU path, same metric

A *step* is one pass of the hot path over the whole synthetic workload (BASELINE.json configs[2]: V=50 000 voxels,
T=200 TRs, E=32 epochs, eps=8): pack the (already normalised, HBM-resident) epochs, then for every voxel row the
correlation GEMM -> Fisher-z + within-subject z-score -> E x E kernel matrix, with the [V, E, E] kernels left resident
in HBM (SURVEY.md §8d).  metric = V * V * E / step time.

N > 1: the symmetric pipeline's row shards (equal trapezoid areas) go to the ranks, the epochs are replicated in every
rank's HBM before the timed region (as after the reference's bcast, preprocessing.py:211-223), and ONE NCCL
reduce-scatter inside the timed step sums the ranks' partial kernels so that every rank ends up with the kernels of the
rows it would cross-validate (voxelselector.py's row partition).  Total work is fixed: "scaling": "strong".

`e2e` is the same metric from HOST buffers to HOST buffers, unpipelined, every copy inside the timed region:
  N = 1: one call of the C-ABI host entry point fcma_host_voxel_kernels_sym per step (pinned host epochs in, pinned host
         kernels out: H2D, packing, kernels, D2H -- synchronous; inside the call the first pass' GEMM follows the upload
         epoch group by epoch group and a pass' kernels are read back under the next pass);
  N > 1: per step every rank uploads ITS share of the epochs (E/N of them) over its own PCIe link, the shares are
         all-gathered over NVLink by the copy engines (CUDA IPC; brainiak_b200/fcma/exchange.py), then pack, kernels,
         reduce-scatter and the read-back of the rank's own kernel rows.
The pipelined variant (copies of step k+1 / k-1 under the kernels of step k) is reported beside it as `e2e.pipelined`.

One JSON line is printed by rank 0.  Extra objects: `roofline` (dominant kernel, measured live with CUDA events),
`kernels` (per-kernel table), `cpu_baseline` (reference path on this box's host cores, bounded sample),
`parity_vs_reference` (three 64-row samples through the UNMODIFIED reference: first pass, a middle pass, ragged tail),
`other_configs` (BASELINE configs[1], [3], [4] with their own roofline and parity sample), `clocks`.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

# the tree bench.py runs from may be read-only: import the project without writing __pycache__ into it
sys.dont_write_bytecode = True

# the reference arm must see all host cores: torchrun exports OMP_NUM_THREADS=1, and OpenBLAS / libgomp read the
# environment when they are loaded, i.e. before anything below imports numpy / scipy
if "--impl" in sys.argv and "reference" in sys.argv:
    _cores = str(len(os.sched_getaffinity(0)))
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = _cores

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(V=50000, T=200, E=32, eps=8)
METRIC = "voxel-pair correlations/sec"
UNIT = "corr/s"
SEED = 1234567890
DUMP_BYTES = 48 << 20       # --dump-outputs: at most this many bytes of kernels


def workload_string(V, T, E, eps):
    return "FCMA VoxelSelector V=%d T=%d E=%d eps=%d (BASELINE configs[2] shape)" % (V, T, E, eps)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="fp16x3")
    ap.add_argument("--voxels", type=int, default=WORKLOAD["V"], help="override V (debug only)")
    ap.add_argument("--block-rows", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the other BASELINE configs")
    ap.add_argument("--no-ipc", action="store_true", help="epoch exchange through NCCL all-gather instead of CUDA IPC copies")
    ap.add_argument("--clock-interval-ms", type=int, default=20, help="nvidia-smi sampling interval")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the [V, E, E] kernels of the last one to DIR/kernels.npy (float32); "
                         "when they exceed %d MB, the rows of a fixed sample (dump_rows: seeded, sorted)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the kernels of the b200 arm")
    return args


def dump_rows(V, E):
    """Rows of the kernels --dump-outputs writes: all of them, or a sample fixed by SEED that fits DUMP_BYTES."""
    n = min(V, DUMP_BYTES // (E * E * 4))
    if n == V:
        return np.arange(V)
    return np.sort(np.random.RandomState(SEED).choice(V, n, replace=False))


def make_epoch(e, T, V, out=None):
    """One synthetic epoch of SURVEY.md §8d (torch CPU generator seeded per epoch, so a rank can generate just its
    share): Gaussian [T, V], a planted common time course in the first V//100 voxels of odd epochs, then the
    reference normalisation (zscore over TRs, ddof=0; / sqrt(T); preprocessing.py:80-84)."""
    import torch
    g = torch.Generator().manual_seed(SEED + e)
    m = torch.randn((T, V), generator=g)
    if e % 2 == 1:
        m[:, : V // 100] += 0.6 * torch.randn((T, 1), generator=g)
    m = (m - m.mean(0, keepdim=True)) / m.std(0, unbiased=False, keepdim=True)
    m = torch.nan_to_num(m) / (T ** 0.5)
    if out is not None:
        out.copy_(m)
        return out
    return m


def make_host_epochs(V, T, E, epochs=None, pin=False):
    import torch
    epochs = list(range(E)) if epochs is None else list(epochs)
    x = torch.empty((len(epochs), T, V), dtype=torch.float32, pin_memory=pin)
    for k, e in enumerate(epochs):
        make_epoch(e, T, V, out=x[k])
    return x


def device_epochs(V, T, E, dev, seed):
    """Synthetic epochs generated ON the device (the big other configs: 12.8 GB at V=100 000, T=500, E=64), same
    recipe; identical on every rank (same seed, same generator)."""
    import torch
    from brainiak_b200.fcma import engine
    g = torch.Generator(device=dev).manual_seed(seed)
    ep = torch.empty((E, T, V), dtype=torch.float32, device=dev)
    for e in range(E):
        torch.randn((T, V), generator=g, out=ep[e])
        if e % 2 == 1:
            ep[e, :, : V // 100] += 0.6 * torch.randn((T, 1), generator=g, device=dev)
    engine.epoch_normalize_(ep)
    return ep


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled every 20 ms from the START of the run (the process needs a few hundred ms before its first
    line, longer than a whole multi-GPU timed region); `window(t0, t1)` then picks the samples whose own timestamps
    fall inside the timed region."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, interval_ms=20):
        self.index = index
        self.interval_ms = int(interval_ms)
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", str(self.interval_ms)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.p = None

    def window(self, t0, t1):
        """Clock record of the samples stamped inside [t0, t1] (time.time() values)."""
        import datetime
        if self.f is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, power, inside = [], 0, set(), [], 0
        for line in self.f.read().splitlines():
            parts = [s.strip() for s in line.split(",")]
            if len(parts) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                c, m, pw = float(parts[2]), float(parts[3]), float(parts[4])
            except ValueError:
                continue
            mx = max(mx, m)
            if ts < t0 - 0.005 or ts > t1 + 0.005:
                continue
            inside += 1
            power.append(pw)
            sm.append(c)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), parts[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples_in_timed_region": inside,
                "power_w_median": float(np.median(power)) if power else None,
                "power_w_max": max(power) if power else None, "sampling": "nvidia-smi -lms %d, samples stamped inside the timed region" % self.interval_ms}

    def close(self):
        self.stop()
        try:
            os.unlink(self.f.name)
        except OSError:
            pass


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ---------------------------------------------------------------------------------------------
def host_threads():
    """Give the reference's BLAS / OpenMP every host core (torchrun exports OMP_NUM_THREADS=1); returns the count."""
    cores = len(os.sched_getaffinity(0))
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:  # pragma: no cover
        pass
    return cores


def reference_selector(raw, eps):
    """(module, unmodified reference VoxelSelector, clf, labels) on host arrays, or None if oracle/_ref is missing."""
    from sklearn import svm
    from oracle import reference
    if not reference.available():
        return None
    E = len(raw)
    labels = [e % 2 for e in range(E)]
    clf = svm.SVC(kernel="precomputed", shrinking=False, C=1)
    m = reference.load()
    vs = m.VoxelSelector(labels, eps, E // eps, raw, voxel_unit=64, process_num=0)
    return m, vs, clf, labels


def reference_task_fn(host_epochs, eps):
    """Returns (fn(start, n) -> seconds for the kernel path a4+a6+a7 of one task, kind, cores)."""
    E, T, V = host_epochs.shape
    raw = [host_epochs[e].numpy() for e in range(E)]
    cores = host_threads()
    ref = reference_selector(raw, eps)
    if ref is not None:
        m, vs, clf, _ = ref

        def fn(start, n):
            t0 = time.perf_counter()
            corr = vs._correlation_computation((start, n))             # voxelselector.py:492
            m.fcma_extension.normalization(corr, eps)                   # voxelselector.py:496
            vs._prepare_for_cross_validation(corr, clf)                 # voxelselector.py:505
            return time.perf_counter() - t0
        return fn, "reference", cores
    from oracle import fcma_oracle as orc

    def fn(start, n):
        t0 = time.perf_counter()
        orc.voxel_block(raw, None, start, n, eps, shrink=True)
        return time.perf_counter() - t0
    return fn, "port", orc.num_threads()


def time_reference_tasks(fn, V, ntasks, budget_s, rows=64, warm=1):
    """Median task time over up to `ntasks` tasks of `rows` voxel rows spread over [0, V) (bounded by budget_s)."""
    for w in range(warm):
        fn(0, rows)
    times, t_start = [], time.perf_counter()
    stride = max(rows, ((V - rows) // max(ntasks, 1)) // rows * rows)
    for k in range(ntasks):
        times.append(fn(min(V - rows, (k * stride) % max(V - rows, 1)), rows))
        if time.perf_counter() - t_start > budget_s and len(times) >= 5:
            break
    return float(np.median(times)), len(times), times


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    V, T, E, eps = args.voxels, WORKLOAD["T"], WORKLOAD["E"], WORKLOAD["eps"]
    host = make_host_epochs(V, T, E)
    fn, kind, cores = reference_task_fn(host, eps)
    rows = 64                                     # the reference's default voxel_unit
    # a "step" of this arm = one task of 64 voxel rows (bounded sample of the same workload); the value is taken from
    # the MEDIAN task time of `steps` tasks after `warmup` tasks, extrapolated by the metric (linear in the
    # number of tasks: every task contracts 64 rows with all V columns of all E epochs)
    med, done, times = time_reference_tasks(fn, V, args.steps, float("inf"), rows=rows, warm=max(args.warmup, 1))
    value = rows * float(V) * E / med
    sample = ("median of %d tasks of %d voxel rows x V=%d x E=%d (kernel path a4+a6+a7 = voxelselector.py:492-505, no CV), "
              "%d BLAS/OpenMP threads" % (done, rows, V, E, cores))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * med,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": workload_string(V, T, E, eps),
                                            "step": "one task of 64 voxel rows against all V columns (bounded sample; "
                                                    "the whole job is V/64 such tasks)",
                                            "threads": cores, "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                             "task_ms_min_median_max": [1e3 * min(times), 1e3 * med, 1e3 * max(times)]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print_json(line)
    return 0


# ---------------------------------------------------------------------------------------------
# parity against the unmodified reference (rank 0, host)
# ---------------------------------------------------------------------------------------------
def parity_samples(raw_list, eps, samples, K_rows, engine, dev, mask_self=False):
    """samples: [(start, n)]; K_rows: dict start -> unshrunk GPU kernels [n, E, E] (device tensors) of those rows.
    The unmodified reference computes the same rows on the host: kernels (after its decimal shrink) and the
    cross-validation accuracies of its own scikit-learn path vs the batched GPU SVM on the GPU kernels.
    mask_self: the self-correlation column (r = 1 +- ulp -> clamp -> pure rounding noise, SURVEY §0.4 / Appendix B) is
    zeroed after the reference's normaliser; the GPU kernels must then come from a FCMA_FLAG_MASK_SELF run."""
    ref = reference_selector(raw_list, eps)
    if ref is None:
        return None
    m, rvs, clf, labels = ref
    E = len(raw_list)
    out = []
    for (s0, n0) in samples:
        corr = rvs._correlation_computation((s0, n0))
        m.fcma_extension.normalization(corr, eps)
        if mask_self:
            for i in range(n0):
                corr[i, :, s0 + i] = 0
        Kref = rvs._prepare_for_cross_validation(corr, clf)          # shrunk kernels [n0, E, E]
        acc_ref = np.array([a for _, a in rvs._do_cross_validation(clf, Kref, (s0, n0))])
        Kg = K_rows[s0].to(dev).clone()
        engine.shrink_kernels_(Kg)
        acc_gpu = engine.svm_cv_precomputed(Kg, labels, E // eps, C=1.0, tol=1e-3)
        Kg = Kg.cpu().numpy()
        out.append({"rows": [int(s0), int(s0 + n0)],
                    "max_abs_dK_over_max_K": float(np.max(np.abs(Kg - Kref)) / np.max(np.abs(Kref))),
                    "cv_accuracy_identical": int(np.sum(acc_gpu == acc_ref)), "cv_accuracy_total": int(n0),
                    "max_abs_d_accuracy": float(np.max(np.abs(acc_gpu - acc_ref)))})
    return out


def sample_starts(V, rows_per_pass, n=64):
    """first pass, a middle pass (its rows receive most of their sums from the column pass) and the ragged tail"""
    mid = (V // 2 // 256) * 256 + 64
    s = [(128, n), (min(mid, V - n), n), (V - n, n)]
    return [x for k, x in enumerate(s) if x not in s[:k]]


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import ctypes as _ct

    import torch
    import torch.distributed as dist
    from brainiak_b200 import _lib
    from brainiak_b200.fcma import engine
    from brainiak_b200.fcma.exchange import EpochExchange
    from brainiak_b200.fcma.voxelselector import VoxelSelector

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg2 = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg2 = dist.new_group(backend="nccl")       # collectives issued from the copy stream (epoch exchange)
    lib = _lib.load()
    _lib.require_device()
    sampler = ClockSampler(local, args.clock_interval_ms)
    atexit.register(sampler.close)      # no nvidia-smi left running, whatever ends the run
    if rank == 0:
        sampler.start()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tf_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "MEASURED_PEAKS.json (hbm_gbs, bf16_tflops_sustained)" if peaks else "fallback 6650 GB/s, 1400 TFLOP/s"

    V, T, E, eps = args.voxels, WORKLOAD["T"], WORKLOAD["E"], WORKLOAD["eps"]
    prec, code = args.precision, _lib.PREC[args.precision]
    flags = 0
    if not (engine.sym_supported(E, eps) and V >= 512 * world):
        raise SystemExit("the bench workload needs the symmetric pipeline (E <= 64, power-of-two eps, V >= 512 per rank)")
    parts = engine.sym_row_partition(V, world)
    start, n = parts[rank]
    block = max(256, (min(args.block_rows, max(n, 1)) + 255) // 256 * 256)
    cv_parts = VoxelSelector.row_partition(V, world)       # the rows each rank cross-validates (and keeps)
    per = cv_parts[0][1]

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    # ---- inputs: every rank holds ITS share of the epochs in pinned host memory (the source of the e2e copies);
    # rank 0 also keeps all epochs on the host for the parity check against the reference
    xch = EpochExchange(E, T, V, dev, group=pg2, nbuf=2, use_ipc=not args.no_ipc)
    e0, ne = xch.share_of()
    host_share = make_host_epochs(V, T, E, epochs=range(e0, e0 + ne), pin=True)
    host_all = None
    if rank == 0 and (world > 1) and not (args.no_cpu_baseline and args.no_e2e):
        host_all = make_host_epochs(V, T, E)
    elif rank == 0:
        host_all = host_share
    epochs = xch.gather(0, host_share)           # replicated in every rank's HBM before the timed region
    cols_variant = bool(lib.fcma_sym_uses_column_pass(code, E, eps, flags))
    work = engine.SymWorkspace(E, V, block, dev, start=start, transposed_copy=not cols_variant)
    Kfull = torch.zeros((world * per, E, E), dtype=torch.float32, device=dev)     # this rank's partial sums, all rows
    Kmine = torch.empty((per, E, E), dtype=torch.float32, device=dev) if world > 1 else None
    Khost = torch.empty((per if world > 1 else V, E, E), dtype=torch.float32, pin_memory=True)
    op_buf = engine.pack_epochs(epochs, None, prec, v_begin=start)
    torch.cuda.synchronize()

    def kernels_step(src, Kdst):
        """pack (only the voxels this shard touches) + symmetric pipeline + reduce-scatter of the partial kernels"""
        op = engine.pack_epochs(src, None, prec, v_begin=start, out=op_buf)
        Kdst[start:].zero_()                 # rows < start are never written by this rank and stay zero
        if n > 0:
            engine.voxel_kernels_sym(op, start, n, eps, flags=flags, work=work, out=Kdst[:V])
        if world > 1:
            dist.reduce_scatter_tensor(Kmine, Kdst)

    # N > 1 e2e: interleaved shares (rank r holds epochs r, r + W, ...) so that contiguous epoch groups complete one after
    # the other and the first passes' GEMMs can follow them (engine.voxel_kernels_sym_grouped); a scratch of two blocks
    e2e_state = {}

    def e2e_step():
        """host -> host, unpipelined: this rank's share H2D + epoch exchange, kernels, read-back of the rank's rows"""
        if world == 1:
            engine.host_voxel_kernels_sym(host_share, eps, precision=prec, flags=flags, device=local,
                                          rows_per_pass=block, out=Khost)
            return
        if not e2e_state:
            e2e_state["cs"] = torch.cuda.Stream(device=dev)
            e2e_state["host"] = make_host_epochs(V, T, E, epochs=xch.interleaved_share(), pin=True)
            e2e_state["work"] = engine.SymWorkspace(E, V, 2 * block, dev, start=start, transposed_copy=not cols_variant)
        cs, main = e2e_state["cs"], torch.cuda.current_stream()
        cs.wait_stream(main)
        src, groups, events = xch.gather_groups(1, e2e_state["host"], stream=cs, ngroups=4)
        Kfull[start:].zero_()
        engine.voxel_kernels_sym_grouped(src, op_buf, start, n, eps, groups, events, flags=flags, work=e2e_state["work"],
                                         out=Kfull[:V])
        dist.reduce_scatter_tensor(Kmine, Kfull)
        Khost.copy_(Kmine, non_blocking=True)

    def timed(nsteps, fn):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.fcma_launch_count()
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(nsteps):
            fn()
        ev1.record()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        # device time between the events; the synchronous host entry point (N = 1 e2e) is also bracketed by wall clock
        ms = torch.tensor([ev0.elapsed_time(ev1), wall], device=dev)
        launches = torch.tensor([float(lib.fcma_launch_count() - l0)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(launches, op=dist.ReduceOp.SUM)
        return float(ms[0]), int(launches[0]), float(ms[1])

    pipe_state = {}

    def timed_e2e_pipelined(nsteps):
        """The same host -> host work with the copies off the critical path: the input of step k+1 (H2D of the share +
        epoch exchange) and the read-back of step k-1 run on a copy stream under the kernels of step k (what a service
        streaming datasets through the engine does).  All copies / collectives of all steps are inside the timed region."""
        main = torch.cuda.current_stream()
        if not pipe_state:
            pipe_state["cs"] = torch.cuda.Stream(device=dev)
            pipe_state["kbuf"] = [Kfull, torch.zeros_like(Kfull)]
            pipe_state["kmine"] = [Kmine, torch.empty_like(Kmine)] if world > 1 else None
        cs, kbuf, kmine = pipe_state["cs"], pipe_state["kbuf"], pipe_state["kmine"]
        ready = [torch.cuda.Event() for _ in range(2)]
        stepdone = [torch.cuda.Event() for _ in range(2)]
        kread = [torch.cuda.Event() for _ in range(2)]
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        cs.wait_event(ev0)
        xch.gather(0, host_share, stream=cs)
        ready[0].record(cs)
        for k in range(nsteps):
            c = k & 1
            if k + 1 < nsteps:
                if k >= 1:
                    # buffer 1-c was packed by step k-1 on EVERY rank once that step's reduce-scatter has completed here
                    cs.wait_event(stepdone[1 - c])
                xch.gather(1 - c, host_share, stream=cs)
                ready[1 - c].record(cs)
            main.wait_event(ready[c])
            if k >= 2:
                main.wait_event(kread[c])                   # the read-back of step k-2 has left the result buffer
            op = engine.pack_epochs(xch.buffers[c], None, prec, v_begin=start, out=op_buf)
            kbuf[c][start:].zero_()
            if n > 0:
                engine.voxel_kernels_sym(op, start, n, eps, flags=flags, work=work, out=kbuf[c][:V])
            res = kbuf[c][:V]
            if world > 1:
                dist.reduce_scatter_tensor(kmine[c], kbuf[c])
                res = kmine[c]
            stepdone[c].record(main)
            cs.wait_event(stepdone[c])
            with torch.cuda.stream(cs):
                Khost.copy_(res, non_blocking=True)
            kread[c].record(cs)
        main.wait_stream(cs)
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms[0])

    # ---- headline: kernel path with the inputs resident in HBM
    for _ in range(max(args.warmup, 3)):
        kernels_step(epochs, Kfull)
    t_begin = time.time()
    ms_total, launches, _ = timed(args.steps, lambda: kernels_step(epochs, Kfull))
    t_end = time.time()
    clocks = None
    if rank == 0:
        time.sleep(0.05)
        clocks = sampler.window(t_begin, t_end)
        sampler.close()
    ms_step = ms_total / args.steps
    corr_total = float(V) * V * E
    value = corr_total / (ms_step * 1e-3)

    # the kernels of the last timed step, before anything below computes into the same buffers
    if args.dump_outputs:
        idx = torch.from_numpy(dump_rows(V, E)).to(dev)
        if world == 1:
            sel = Kfull[idx]
        else:
            lo = rank * per                 # Kmine holds rows [lo, lo + per); the other ranks add zeros
            mine = (idx >= lo) & (idx < lo + per)
            sel = torch.zeros((len(idx), E, E), dtype=torch.float32, device=dev)
            sel[mine] = Kmine[idx[mine] - lo]
            dist.reduce(sel, dst=0)
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "kernels.npy"), sel.cpu().numpy())
        del sel

    # per-rank time of the shard alone (no collective): the load balance of the equal-area partition
    balance = None
    if world > 1:
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier(device_ids=[local])
        a.record()
        for _ in range(2):
            engine.pack_epochs(epochs, None, prec, v_begin=start, out=op_buf)
            Kfull[start:].zero_()
            engine.voxel_kernels_sym(op_buf, start, n, eps, flags=flags, work=work, out=Kfull[:V])
        b.record()
        torch.cuda.synchronize()
        mine = torch.tensor([a.elapsed_time(b) / 2], device=dev)
        allms = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allms, mine)
        balance = {"shard_ms_per_rank": [round(float(x[0]), 3) for x in allms],
                   "shard_rows": [[s, s + m] for s, m in parts]}

    # ---- e2e: host -> host
    e2e = None
    if not args.no_e2e:
        e2e_step()
        ne_steps = max(2, min(args.steps, 4))
        ms_dev, _, ms_wall = timed(ne_steps, e2e_step)
        ms_seq = (ms_wall if world == 1 else ms_dev) / ne_steps
        # the host -> host result against the kernel path's (same inputs): both must be the same kernels
        torch.cuda.synchronize()
        Kh = Khost.to(dev)
        kernels_step(epochs, Kfull)
        Kd = Kmine if world > 1 else Kfull[:V]
        e2e_check = torch.stack([(Kh - Kd).abs().max(), Kd.abs().max()])
        if world > 1:
            dist.all_reduce(e2e_check, op=dist.ReduceOp.MAX)
        e2e_dk = float(e2e_check[0] / e2e_check[1])
        del Kh
        npipe = max(8, 2 * args.steps)      # the first copy-in and the last read-back cannot hide: amortise them
        timed_e2e_pipelined(2)
        ms_pipe = timed_e2e_pipelined(npipe) / npipe
        share_bytes = int(ne) * T * V * 4
        e2e = {"value": corr_total / (ms_seq * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(E) * T * V * 4, "d2h_bytes_per_step": int(V) * E * E * 4,
               "h2d_bytes_per_step_per_rank": share_bytes, "d2h_bytes_per_step_per_rank": int(Khost.numel()) * 4,
               "ms_per_step": ms_seq, "steps": ne_steps,
               "max_abs_dK_over_max_K_vs_kernel_path": e2e_dk,
               "path": ("one fcma_host_voxel_kernels_sym call per step (C ABI, include/fcma_b200.h): pinned host epochs -> H2D "
                        "-> pack -> symmetric pipeline -> D2H -> pinned host kernels, synchronous, timed by wall clock"
                        if world == 1 else
                        "per step and rank: H2D of the rank's E/N epochs (interleaved share) over its own PCIe link -> all-gather of "
                        "the shares over NVLink (%s), completing in 4 contiguous epoch groups -> per group: pack + GEMMs of the "
                        "first two passes (fcma_voxel_kernels_sym_grouped), then the rest of the symmetric pipeline -> NCCL "
                        "reduce-scatter -> D2H of the rank's own kernel rows; one step at a time, CUDA events, max over ranks"
                        % xch.mode),
               "epoch_exchange": xch.mode,
               "pipelined": {"value": corr_total / (ms_pipe * 1e-3), "unit": UNIT, "ms_per_step": ms_pipe, "steps": npipe,
                             "how": "copy stream + double buffers: input of step k+1 and read-back of step k-1 under the kernels "
                                    "of step k; every copy and collective of all steps inside the timed region"}}

    # ---- roofline of the step's kernels, measured live with CUDA events on the launch stream (rank 0's shard)
    roofline, kernels = None, None
    if rank == 0:
        planes = lib.fcma_operand_planes(code)
        kp = lib.fcma_operand_kp(code, T)
        op_bytes = lib.fcma_operand_bytes(code, E, T, V)
        nprod = 3 if planes == 2 else 1
        rpp = int(lib.fcma_sym_rows_per_pass(code, E, eps, flags, V, start, work.buf.numel()))
        kernels, summary = sym_kernel_table(lib, engine, torch, op_buf, start, n, V, T, E, eps, flags, work, Kfull[:V], rpp,
                                            cols_variant, op_bytes, nprod, kp, hbm_peak, tf_peak)
        dominant = max(kernels, key=lambda k: kernels[k]["ms"])
        traffic, traffic_src = None, None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            tag = "symcols:rows%d" % min(rpp, 4096)
            ent = tr.get("%s:%s:%s" % (dominant.split(" ")[0], prec, tag)) or \
                tr.get("%s:%s:%s" % (dominant.split(" ")[0].replace("umma2", "umma"), prec, tag))
            if isinstance(ent, dict):
                traffic = ent["ratio"] * kernels[dominant]["algorithmic_bytes"]
                traffic_src = ("static: dram bytes / algorithmic bytes = %.3f of the first (largest) launch under ncu --set full "
                               "(profiles/traffic.json), applied to the average launch" % ent["ratio"])
        except Exception:
            pass
        ach = kernels[dominant]["hbm_gbs"]
        # step level: bytes the design moves per step (block written once, read by the row pass and by the column pass,
        # operand read once per pass) against the HBM peak, and the delivered flops (SURVEY §8d: 2T + E + 1 per
        # correlation) against the sustained tensor peak
        flop_per_corr = 2.0 * T + E + 1
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peak_src, "launch_ms": kernels[dominant]["ms"],
                    "launches_per_step": summary["passes"], "rows_per_launch": rpp,
                    "algorithmic_bytes_per_launch": kernels[dominant]["algorithmic_bytes"],
                    "tensor": {"delivered_tflops": value * flop_per_corr / 1e12, "peak_tflops": tf_peak,
                               "frac": value * flop_per_corr / 1e12 / tf_peak,
                               "flop_per_corr": flop_per_corr, "note": "SURVEY §8d delivered flops (one product, symmetric halves not "
                               "double counted) / sustained cuBLAS bf16 peak; the fp32-faithful split EXECUTES 3 products"},
                    "step": {"algorithmic_bytes": summary["step_bytes"] * (world if world > 1 else 1),
                             "hbm_frac": summary["step_bytes"] / (summary["sum_ms"] * 1e-3) / 1e9 / hbm_peak,
                             "note": "bytes the two-pass design moves per step (rank 0's shard) / (sum of its kernel times x HBM peak)"},
                    "pipeline": "symmetric (blocks on/above the diagonal stored once, read row-wise and column-wise)" if cols_variant
                                else "symmetric (blocks on/above the diagonal, each stored twice)"}

    # ---- parity against the UNMODIFIED reference at the full shape: three 64-row samples
    parity = None
    samples = sample_starts(V, block)
    if not args.no_cpu_baseline or world > 1:
        kernels_step(epochs, Kfull)
        rows = {}
        if world > 1:
            # the reduce-scattered result: sample rows live on the rank that owns them
            for (s0, n0) in samples:
                owner = min(s0 // per, world - 1)
                buf = torch.zeros((n0, E, E), device=dev)
                if rank == owner:
                    buf.copy_(Kmine[s0 - owner * per: s0 - owner * per + n0])
                dist.broadcast(buf, src=owner)
                rows[s0] = buf
        else:
            rows = {s0: Kfull[s0:s0 + n0].clone() for (s0, n0) in samples}
        if rank == 0 and host_all is not None:
            host_threads()
            raw_list = [host_all[e].numpy() for e in range(E)]
            res = parity_samples(raw_list, eps, samples, rows, engine, dev)
            if res is not None:
                parity = {"vs": "unmodified reference (oracle/_ref) on the host, same inputs; kernels after the decimal shrink, "
                                "CV accuracies of its scikit-learn path vs the batched GPU SVM",
                          "pipeline": "symmetric, %d GPU%s%s" % (world, "s" if world > 1 else "",
                                                                 " (after the NCCL reduce-scatter)" if world > 1 else ""),
                          "samples": res,
                          "max_abs_dK_over_max_K": max(r["max_abs_dK_over_max_K"] for r in res),
                          "cv_accuracy_identical": sum(r["cv_accuracy_identical"] for r in res),
                          "cv_accuracy_total": sum(r["cv_accuracy_total"] for r in res)}

    # ---- the public API end to end: VoxelSelector.run(clf) incl. the batched GPU SVM cross-validation
    run_api = None
    if rank == 0 and world == 1 and not args.no_e2e:
        from sklearn import svm as _svm
        raw_list = [host_all[e].numpy() for e in range(E)]
        labels = [e % 2 for e in range(E)]
        clf = _svm.SVC(kernel="precomputed", shrinking=False, C=1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        vs = VoxelSelector(labels, eps, E // eps, raw_list, voxel_unit=64, process_num=0, precision=prec,
                           block_rows=block)
        vs._work = work
        res = vs.run(clf)
        torch.cuda.synchronize()
        t_run = time.perf_counter() - t0
        top = sorted(v for v, _ in res[: V // 100])
        run_api = {"seconds": t_run, "value": corr_total / t_run, "unit": UNIT,
                   "what": "VoxelSelector(labels, eps, folds, raw_data).run(SVC(kernel='precomputed')) from host numpy "
                           "epochs to the sorted (voxel, accuracy) list: H2D + pack + kernels + decimal shrink + "
                           "batched GPU SVM cross-validation (%d voxels x %d folds)" % (V, E // eps),
                   "planted_voxels_in_top_1pct": int(sum(1 for v in top if v < V // 100)), "top_1pct_size": V // 100}

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        fn, kind, cores = reference_task_fn(host_all, eps)
        med, done, times = time_reference_tasks(fn, V, 20, 25.0)
        cpu_baseline = {"value": 64 * float(V) * E / med, "unit": UNIT, "cores": cores, "kind": kind,
                        "sample": "median of %d tasks of 64 voxel rows x V=%d x E=%d, kernel path a4+a6+a7 "
                                  "(reference voxelselector.py:492-505), no CV; %d threads" % (done, V, E, cores),
                        "task_ms_min_median_max": [1e3 * min(times), 1e3 * med, 1e3 * max(times)]}

    # ---- the other BASELINE.json configs on the same path, each with its own roofline and parity sample
    others = None
    if not args.no_others:
        del work, op_buf
        e2e_state.clear()
        torch.cuda.empty_cache()
        others = other_configs(args, lib, engine, torch, dist, dev, rank, world, local, hbm_peak, tf_peak)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None,
                "dtype": {"fp16x3": "f16x3 (hi/lo split, f32 accumulate)", "tf32x3": "tf32x3 (hi/lo split, f32 accumulate)",
                          "bf16x3": "bf16x3", "tf32": "tf32", "bf16": "bf16"}.get(prec, prec),
                "data": "synthetic",
                "config": {"workload": workload_string(V, T, E, eps),
                           "precision": prec + (" (3-product hi/lo split, fp32-faithful: |dr| <= 1e-6)" if prec in ("tf32x3", "fp16x3") else ""),
                           "parallelism": "rows%d" % world, "rows_per_pass": block,
                           "pipeline": "symmetric self-correlation: blocks on/above the diagonal contracted once, used for row and "
                                       "column voxels; shards = equal-area row ranges",
                           "l2": "inputs_exceed_l2 (operand %.1f GB, correlation block %.1f GB per pass)"
                                 % (lib.fcma_operand_bytes(code, E, T, V) / 1e9, lib.fcma_work_bytes_per_row(E, V) * block / 1e9),
                           "step": "pack + corr GEMM + Fisher/z-score + kernel build for all V rows"
                                   + ("; epochs replicated in every rank's HBM beforehand, one NCCL reduce-scatter of the partial "
                                      "[V,E,E] kernels inside the step (every rank keeps the rows it cross-validates)" if world > 1 else "")},
                "gpu_launches": launches, "e2e": e2e, "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu_baseline,
                "voxel_selection_run": run_api, "parity_vs_reference": parity, "load_balance": balance,
                "other_configs": others, "clocks": clocks}
        print_json(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def sym_kernel_table(lib, engine, torch, op, start, n, V, T, E, eps, flags, work, K, rpp, cols_pass, op_bytes, nprod, kp,
                     hbm_peak, tf_peak, reps=2):
    """Live per-kernel times (CUDA events inside the C pipeline, fcma_timing_*) of the launches of one symmetric step over
    rows [start, start+n), with the algorithmic bytes of each kernel: GEMM = 4 B per stored correlation + operand read
    once; row pass = the block read once; column pass = the block right of the diagonal part read once."""
    import ctypes as _ct
    esz = 4.0
    launches_desc, pass2, rows_el = [], 0.0, 0.0
    for a in range(start, start + n, rpp):
        nn = min(rpp, start + n - a)
        colsA, rowsB = V - a, V - a - nn
        nt, t256 = -(-nn // 256), -(-colsA // 256)
        stored = float(nn) * colsA + (0.0 if cols_pass else float(rowsB) * nn)
        launches_desc.append((stored, colsA, nt * (nt + 1) // 2 + (t256 - nt) * nt))
        pass2 += float(nn) * colsA + float(rowsB) * nn
        rows_el += float(nn) * colsA

    def one_pass():
        K[start:].zero_()
        engine.voxel_kernels_sym(op, start, n, eps, flags=flags, work=work, out=K)
    one_pass()
    torch.cuda.synchronize()
    lib.fcma_timing_enable(1)
    for _ in range(reps):
        one_pass()
    torch.cuda.synchronize()
    g_ms, s_ms, s2_ms = _ct.c_double(0), _ct.c_double(0), _ct.c_double(0)
    npass = lib.fcma_timing_read3(_ct.byref(g_ms), _ct.byref(s_ms), _ct.byref(s2_ms))
    lib.fcma_timing_enable(0)
    assert npass == reps * len(launches_desc), (npass, len(launches_desc))
    nl = float(len(launches_desc))
    tg, ts, ts2 = g_ms.value / npass, s_ms.value / npass, s2_ms.value / npass
    corr_launch = sum(d[0] for d in launches_desc) * E / nl
    opread = sum(d[1] for d in launches_desc) / nl / V * op_bytes
    tiles = sum(d[2] for d in launches_desc) / nl * E
    rows_bytes = esz * rows_el * E / nl
    second_bytes = esz * (pass2 - rows_el) * E / nl
    alg = esz * corr_launch + opread
    flop_exec = nprod * 2.0 * kp * tiles * 65536.0
    kernels = {
        "k_corr_umma2": {"ms": tg, "algorithmic_bytes": alg, "hbm_gbs": alg / (tg * 1e-3) / 1e9,
                         "tensor_tflops_executed": flop_exec / (tg * 1e-3) / 1e12,
                         "tensor_executed_frac_of_bf16_sustained": flop_exec / (tg * 1e-3) / 1e12 / tf_peak},
        "k_norm_syrk": {"ms": ts, "algorithmic_bytes": rows_bytes, "hbm_gbs": rows_bytes / (ts * 1e-3) / 1e9}}
    if ts2 > 0:
        name = "k_norm_syrk_cols" if cols_pass else "k_norm_syrk (transposed block)"
        kernels[name] = {"ms": ts2, "algorithmic_bytes": second_bytes, "hbm_gbs": second_bytes / (ts2 * 1e-3) / 1e9}
    for kd in kernels.values():
        kd["frac_of_hbm_peak"] = kd["hbm_gbs"] / hbm_peak
        kd["share_of_step"] = kd["ms"] / (tg + ts + ts2)
        kd["ms_per_step"] = kd["ms"] * nl
    step_bytes = (alg + rows_bytes + second_bytes) * nl
    return kernels, {"passes": int(nl), "step_bytes": step_bytes, "sum_ms": (tg + ts + ts2) * nl}


def other_configs(args, lib, engine, torch, dist, dev, rank, world, local, hbm_peak, tf_peak):
    """BASELINE.json configs[1] (V=30 000 T=200 E=16, 1 GPU), configs[3] (V=100 000 T=500 E=64, row shards over all
    ranks) and configs[4] (Classifier kernel, V=50 000 E=32, 1 GPU): device-timed step, per-kernel roofline and one parity
    sample through the unmodified reference each.  Inputs are generated on the device (identical on every rank)."""
    from brainiak_b200 import _lib
    from brainiak_b200.fcma.voxelselector import VoxelSelector
    out = {}
    prec = args.precision
    code = _lib.PREC[prec]

    def run_cfg(name, V, T, E, eps, rows_req, sharded, ref_rows=32):
        w = world if sharded else 1
        if not sharded and rank != 0:
            return
        start, n = engine.sym_row_partition(V, w)[rank if sharded else 0]
        ep = device_epochs(V, T, E, dev, seed=SEED + 17 * E + T)
        op = engine.pack_epochs(ep, None, prec, v_begin=start)
        cols = bool(lib.fcma_sym_uses_column_pass(code, E, eps, 0))
        per_row = (1 if cols else 2) * lib.fcma_work_bytes_per_row(E, V - start)
        free, _ = torch.cuda.mem_get_info(dev)
        rows = max(256, min(rows_req, (n + 255) // 256 * 256, int((free - (6 << 30)) // per_row) // 256 * 256))
        work = engine.SymWorkspace(E, V, rows, dev, start=start, transposed_copy=not cols)
        per = VoxelSelector.row_partition(V, w)[0][1]
        K = torch.zeros((w * per, E, E), dtype=torch.float32, device=dev)
        Kmine = torch.empty((per, E, E), dtype=torch.float32, device=dev) if w > 1 else None

        def step():
            engine.pack_epochs(ep, None, prec, v_begin=start, out=op)
            K[start:].zero_()
            engine.voxel_kernels_sym(op, start, n, eps, work=work, out=K[:V])
            if w > 1:
                dist.reduce_scatter_tensor(Kmine, K)
        step()
        if w > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 2
        a.record()
        for _ in range(reps):
            step()
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / reps], device=dev)
        if w > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms[0])
        corr_total = float(V) * V * E
        # parity sample: the reference on the host for ref_rows rows of the tail of rank 0's shard ... of the whole job
        samples = [(min(V - ref_rows, (V // 2 // 256) * 256 + 32), ref_rows)]
        rows_k = {}
        for (s0, n0) in samples:
            if w > 1:
                owner = min(s0 // per, w - 1)
                buf = torch.zeros((n0, E, E), device=dev)
                if rank == owner:
                    buf.copy_(Kmine[s0 - owner * per: s0 - owner * per + n0])
                dist.broadcast(buf, src=owner)
                rows_k[s0] = buf
            else:
                rows_k[s0] = K[s0:s0 + n0].clone()
        # T > 256: second, untimed run with the self column masked (see parity_note below)
        masked_rows = None
        if T > 256 and (not args.no_cpu_baseline or w > 1):
            engine.pack_epochs(ep, None, prec, v_begin=start, out=op)
            K[start:].zero_()
            engine.voxel_kernels_sym(op, start, n, eps, flags=_lib.FLAG_MASK_SELF, work=work, out=K[:V])
            masked_rows = {}
            if w > 1:
                dist.reduce_scatter_tensor(Kmine, K)
            for (s0, n0) in samples:
                if w > 1:
                    owner = min(s0 // per, w - 1)
                    buf = torch.zeros((n0, E, E), device=dev)
                    if rank == owner:
                        buf.copy_(Kmine[s0 - owner * per: s0 - owner * per + n0])
                    dist.broadcast(buf, src=owner)
                    masked_rows[s0] = buf
                else:
                    masked_rows[s0] = K[s0:s0 + n0].clone()
        entry = None
        if rank == 0:
            planes = lib.fcma_operand_planes(code)
            rpp = int(lib.fcma_sym_rows_per_pass(code, E, eps, 0, V, start, work.buf.numel()))
            kern, summ = sym_kernel_table(lib, engine, torch, op, start, n, V, T, E, eps, 0, work, K[:V], rpp, cols,
                                          lib.fcma_operand_bytes(code, E, T, V), 3 if planes == 2 else 1,
                                          lib.fcma_operand_kp(code, T), hbm_peak, tf_peak, reps=1)
            dom = max(kern, key=lambda k: kern[k]["ms"])
            flop_per_corr = 2.0 * T + E + 1
            entry = {"workload": "FCMA VoxelSelector V=%d T=%d E=%d eps=%d" % (V, T, E, eps), "n_gpus": w,
                     "ms_per_step": ms, "value": corr_total / (ms * 1e-3), "unit": UNIT, "rows_per_pass": rpp,
                     "pipeline": "symmetric, " + ("column pass over the stored block" if cols else
                                                  "transposed copy of every block + row pass (E > 32)"),
                     "roofline": {"kernel": dom, "bound": "hbm", "achieved": kern[dom]["hbm_gbs"], "peak": hbm_peak,
                                  "unit": "GB/s", "frac": kern[dom]["frac_of_hbm_peak"],
                                  "tensor_frac": corr_total / (ms * 1e-3) * flop_per_corr / 1e12 / tf_peak,
                                  "step_hbm_frac": summ["step_bytes"] / (summ["sum_ms"] * 1e-3) / 1e9 / hbm_peak},
                     "kernels": {k: {"ms_per_step": v["ms_per_step"], "frac_of_hbm_peak": v["frac_of_hbm_peak"]} for k, v in kern.items()}}
            if not args.no_cpu_baseline or w > 1:
                host_threads()
                hostep = ep.cpu()
                raw_list = [hostep[e].numpy() for e in range(E)]
                res = parity_samples(raw_list, eps, samples, rows_k, engine, dev)
                entry["parity_vs_reference"] = res[0] if res else None
                if masked_rows is not None:
                    resm = parity_samples(raw_list, eps, samples, masked_rows, engine, dev, mask_self=True)
                    entry["parity_vs_reference_self_column_masked"] = resm[0] if resm else None
                    entry["parity_note"] = ("T > 256: the reference's sgemm blocks the time axis, so its r(i,i) = 1 +- ulp pattern is no "
                                            "longer the sequential FMA chain the packed operand reproduces; the self column is pure "
                                            "rounding noise amplified by the z-score (one column of V: up to ~(eps-1)/V of a kernel "
                                            "entry, SURVEY Appendix B) -- with that column zeroed on both sides the kernels agree")
                del hostep, raw_list
            out[name] = entry
        del work, K, op, ep
        torch.cuda.empty_cache()

    run_cfg("configs[1] V=30000 T=200 E=16 (1 GPU)", 30000, 200, 16, 8, 4096, sharded=False)
    if os.environ.get("FCMA_BENCH_SKIP_CONFIG3") != "1":
        run_cfg("configs[3] V=100000 T=500 E=64 (%d GPU%s)" % (world, "s" if world > 1 else ""), 100000, 500, 64, 8,
                4096, sharded=True, ref_rows=16)
    if rank == 0:
        # configs[4]: Classifier precomputed corr-kernel matrix, V=50 000 E=32: ONE [E, E] kernel = sum over all voxel rows
        V, T, E, eps = 50000, 200, 32, 8
        ep = device_epochs(V, T, E, dev, seed=SEED + 4)
        op = engine.pack_epochs(ep, None, prec)
        work = engine.SymWorkspace(E, V, 4096, dev, transposed_copy=False)
        Kc = torch.zeros((E, E), dtype=torch.float32, device=dev)
        engine.classifier_kernel(op, op, 0, V, eps, work=work, out=Kc)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        Kc.zero_()
        engine.classifier_kernel(op, op, 0, V, eps, work=work, out=Kc)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        # live per-kernel times of the classifier path: per pass one symmetric GEMM (block stored once) and the row passes
        # over it (diagonal square + the columns right of it = the block read ONCE); no column-direction pass
        import ctypes as _ct
        lib.fcma_timing_enable(1)
        Kc2 = torch.zeros((E, E), dtype=torch.float32, device=dev)
        engine.classifier_kernel(op, op, 0, V, eps, work=work, out=Kc2)
        torch.cuda.synchronize()
        g_ms, s_ms = _ct.c_double(0), _ct.c_double(0)
        npass = lib.fcma_timing_read(_ct.byref(g_ms), _ct.byref(s_ms))
        lib.fcma_timing_enable(0)
        code = _lib.PREC[prec]
        blk = sum(float(min(4096, V - a)) * -(-(V - a) // 256) * 256 for a in range(0, V, 4096)) * E * 4.0     # bytes of all blocks
        opb = sum(float(V - a) / V for a in range(0, V, 4096)) * lib.fcma_operand_bytes(code, E, T, V)
        kern = {"k_corr_umma2": {"ms_per_step": g_ms.value, "frac_of_hbm_peak": (blk + opb) / (g_ms.value * 1e-3) / 1e9 / hbm_peak},
                "k_norm_syrk (square + rest)": {"ms_per_step": s_ms.value, "frac_of_hbm_peak": blk / (s_ms.value * 1e-3) / 1e9 / hbm_peak}}
        dom = max(kern, key=lambda k: kern[k]["ms_per_step"])
        # parity: K_classifier == sum of the per-voxel kernels (fp64 sum on the GPU), and sampled per-voxel kernels against
        # the reference's own (the full reference run of this config is ~0.5 h of CPU)
        Kv = torch.zeros((V, E, E), dtype=torch.float32, device=dev)
        engine.voxel_kernels_sym(op, 0, V, eps, work=work, out=Kv)
        Ksum = Kv.to(torch.float64).sum(0)
        ent = {"workload": "FCMA Classifier precomputed corr-kernel matrix V=%d T=%d E=%d eps=%d (one [E,E] kernel)" % (V, T, E, eps),
               "n_gpus": 1, "ms_per_step": ms, "value": float(V) * V * E / (ms * 1e-3), "unit": UNIT, "passes": int(npass),
               "pipeline": "fcma_classifier_kernel_sym: symmetric GEMM + row passes only (diagonal squares once, the blocks right "
                           "of them twice), fp64 accumulation",
               "max_abs_dK_vs_fp64_sum_of_voxel_kernels": float((Kc.to(torch.float64) - Ksum).abs().max() / Ksum.abs().max()),
               "kernels": kern,
               "roofline": {"kernel": dom, "bound": "hbm", "achieved": kern[dom]["frac_of_hbm_peak"] * hbm_peak, "peak": hbm_peak,
                            "unit": "GB/s", "frac": kern[dom]["frac_of_hbm_peak"],
                            "step_hbm_frac": (2 * blk + opb) / ((g_ms.value + s_ms.value) * 1e-3) / 1e9 / hbm_peak}}
        if not args.no_cpu_baseline:
            host_threads()
            hostep = ep.cpu()
            raw_list = [hostep[e].numpy() for e in range(E)]
            s0 = (V // 2 // 256) * 256 + 32
            res = parity_samples(raw_list, eps, [(s0, 32)], {s0: Kv[s0:s0 + 32].clone()}, engine, dev)
            ent["parity_vs_reference_voxel_kernels"] = res[0] if res else None
        out["configs[4] Classifier kernel V=50000 E=32 (1 GPU)"] = ent
    return out if rank == 0 else None


def main():
    args = parse()
    # Exactly ONE line may reach stdout (the JSON): libraries (NCCL's version banner, warnings) write
    # to fd 1 as well, so fd 1 is pointed at stderr for the whole run and the JSON line goes to the
    # saved original stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real_stdout, "w")
    global print_json

    def print_json(obj):
        out.write(json.dumps(obj) + "\n")
        out.flush()
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


def print_json(obj):      # replaced in main()
    print(json.dumps(obj), flush=True)


if __name__ == "__main__":
    sys.exit(main())
