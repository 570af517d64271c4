#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json.

Headline (default, `--config cfg2`): `MulticlassConfusionMatrix(num_classes=1000)` updated with [65536, 1000] bf16 logits
(configs[1]); one "step" = one `update()` over one batch = 65,536,000 metric-updates.

    python bench.py --gpus N --steps K --warmup W            # ours (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU implementation on the host cores
    python bench.py --config cfg3|cfg4|cfg5 [...]            # the other BASELINE.json configs, same line format
    python bench.py --steps K --warmup W --dump-outputs DIR  # + DIR/confmat.npy: what the last timed step computed

Prints ONE JSON line (rank 0).  See DESIGN.md §4 for how each field is obtained.  The default cfg2 line also carries
  config.sync   the cross-rank state sync of the [C, C] confusion matrix, timed on its own (N > 1)
  config.cfg5   MetricCollection([MulticlassF1Score, MulticlassAUROC], C=1000): updates + compute incl. the class-sharded
                exchange, with parity checks (N >= 1)
  aten_gpu_baseline   the stock ATen op chain the reference executes, timed on the SAME B200 (SURVEY.md §2.2's bar)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_ROWS, N_CLASSES = 65536, 1000
UNITS_PER_STEP = N_ROWS * N_CLASSES
# algorithmic bytes of ONE update launch (SURVEY.md §8(d)): logits N*C*2 + target N*8 + one 8-byte counter RMW per row
ALGO_BYTES_PER_LAUNCH = N_ROWS * N_CLASSES * 2 + N_ROWS * 8 + N_ROWS * 8
METRIC = "metric-updates/sec (batch x classes)"
UNIT = "updates/s"
N_ROT = int(os.environ.get("MB200_BENCH_NROT", "16"))  # distinct device batches cycled through (each 131 MB)
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
_REASONS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons through NVML, sampled by a CHILD PROCESS (benchmarks/_clock_sampler.py) so that the
    sampling never takes the interpreter lock away from the launch loop; `window()` records wall-clock brackets of the timed
    regions, `stop()` keeps the samples that fall inside them."""

    def __init__(self, index: int) -> None:
        self.windows = {}
        self.proc = None
        try:
            self.proc = subprocess.Popen([sys.executable, os.path.join(ROOT, "benchmarks", "_clock_sampler.py"), str(index)],
                                         stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def wait_ready(self) -> None:
        if self.proc is not None:
            try:
                self.proc.stdout.readline()
            except Exception:
                self.proc = None

    def window(self, name: str, t0: float, t1: float) -> None:
        self.windows[name] = (t0, t1)

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.stdin.close()
            data = json.loads(self.proc.stdout.readline())
            self.proc.wait(timeout=10)
        except Exception:
            return out
        out["sm_max_mhz"] = data.get("max_mhz")
        samples = data.get("samples") or []

        def inside(names):
            return [s for s in samples if any(self.windows[n][0] <= s[0] <= self.windows[n][1] for n in names if n in self.windows)]

        picked, which = inside(["value"]), "the K timed update steps"
        if len(picked) < 3:  # a 20-step region lasts ~0.5 ms: widen to every device-timed region of this run
            picked, which = inside(list(self.windows)), "all timed regions of this run (" + ", ".join(self.windows) + ")"
        if picked:
            out["sm_mhz"] = statistics.median(s[1] for s in picked)
            bits = 0
            for s in picked:
                bits |= s[2]
            out["reasons"] = sorted(k for k, v in _REASONS.items() if bits & v)
        out["samples"] = len(picked)
        out["window"] = which
        out["sampler"] = "separate process, NVML, back-to-back queries"
        return out


def make_batch(seed: int):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(N_ROWS, N_CLASSES, generator=g).bfloat16()
    target = torch.randint(0, N_CLASSES, (N_ROWS,), generator=g)
    return logits, target


def have_reference() -> bool:
    return os.path.isdir(os.path.join(REF_DIR, "torchmetrics"))


def import_reference():
    """The UNMODIFIED reference installed under baseline/_ref (pip --no-deps --target, DESIGN.md §4).  Its one missing
    dependency, `lightning_utilities` (4 symbols), is served by the labelled stand-in of tests/golden/_standins when the real
    package is not installed."""
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        import lightning_utilities  # noqa: F401
    except Exception:
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden", "_standins"))
    import torchmetrics

    assert os.path.abspath(torchmetrics.__file__).startswith(REF_DIR), torchmetrics.__file__
    return torchmetrics


# --------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU implementation on the host cores
# --------------------------------------------------------------------------------------------------------------
def cpu_update_fn():
    """(callable(logits, target) -> None, kind, description): one MulticlassConfusionMatrix.update on CPU tensors."""
    if have_reference():
        tm = import_reference()
        metric = tm.classification.MulticlassConfusionMatrix(num_classes=N_CLASSES, validate_args=False)
        return metric.update, "reference", ("the unmodified reference (baseline/_ref, TorchMetrics "
                                            f"{tm.__version__}) MulticlassConfusionMatrix(validate_args=False).update on CPU tensors")
    from oracle.torch_cpu_chain import multiclass_confmat_update_cpu

    confmat = torch.zeros(N_CLASSES, N_CLASSES, dtype=torch.long)
    return (lambda lg, tg: multiclass_confmat_update_cpu(confmat, lg, tg, N_CLASSES)), "port", \
        "reference CPU op chain argmax->t*C+p->bincount->+= restated in oracle/torch_cpu_chain.py (baseline/_ref absent)"


def time_cpu_chain(logits, target, rows: int, steps: int, warmup: int):
    """Per-step wall times of the reference's CPU update at the best thread count of this host: every candidate count gets
    1 warm-up + 5 timed calls, the one with the smallest MINIMUM wins (medians flip between runs on a busy host)."""
    update, kind, what = cpu_update_fn()
    lg, tg = logits[:rows], target[:rows]
    ncpu = os.cpu_count() or 1
    calib = {}
    for cand in sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}):
        torch.set_num_threads(cand)
        update(lg, tg)
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            update(lg, tg)
            ts.append(time.perf_counter() - t0)
        calib[cand] = min(ts)
    best_t = min(calib, key=calib.get)
    torch.set_num_threads(best_t)
    for _ in range(warmup):
        update(lg, tg)
    per_step = []
    for _ in range(steps):
        t0 = time.perf_counter()
        update(lg, tg)
        per_step.append(time.perf_counter() - t0)
    return {"total_s": sum(per_step), "min_s": min(per_step), "median_s": statistics.median(per_step),
            "threads": best_t, "kind": kind, "what": what,
            "calibration_ms": {str(k): round(v * 1e3, 3) for k, v in calib.items()}}


def run_reference(args) -> dict:
    if args.config != "cfg2":
        from benchmarks import run_configs

        return run_configs.reference_line(args)
    logits, target = make_batch(0)
    # bound the whole run to roughly a minute: full batches cost 5-50 ms each depending on the host
    budget_s, est_full = 60.0, 0.06
    rows = N_ROWS
    while rows > 1024 and (args.steps + args.warmup) * est_full * rows / N_ROWS > budget_s:
        rows //= 2
    r = time_cpu_chain(logits, target, rows, args.steps, args.warmup)
    # `value` from the MEDIAN step: a 128-core shared host throws 100 ms outliers into a 5 ms step, and the mean over 20
    # steps then swings 5x between runs.  The median is the reference at its steady best — the conservative denominator for
    # every speed-up quoted against it; the total-time figure is kept beside it.
    ups = rows * N_CLASSES / r["median_s"]
    sample = (f"{args.steps} update() calls on the first {rows} rows of the seed-0 [65536,1000] bf16 batch; value = units / "
              f"median step ({r['median_s'] * 1e3:.2f} ms; mean {r['total_s'] / args.steps * 1e3:.2f} ms)")
    return {
        "impl": "reference",
        "metric": METRIC, "value": ups, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["median_s"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "MulticlassConfusionMatrix(num_classes=1000).update, [65536,1000] bf16 logits + int64 target",
                   "rows_per_step": rows, "device": "cpu", "what": r["what"],
                   "value_from_total_time": rows * N_CLASSES * args.steps / r["total_s"],
                   "ms_per_step_min": r["min_s"] * 1e3, "ms_per_step_median": r["median_s"] * 1e3,
                   "thread_calibration_ms": r["calibration_ms"]},
        "cpu_baseline": {"value": ups, "unit": UNIT, "cores": r["threads"], "kind": r["kind"], "sample": sample},
        "e2e": {"value": ups, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


# --------------------------------------------------------------------------------------------------------------
# the stock ATen op chain of the reference on the SAME GPU (SURVEY.md §2.2: the bar for every new kernel)
# --------------------------------------------------------------------------------------------------------------
def aten_gpu_cfg2(dev, dev_batches, steps: int) -> dict:
    if have_reference():
        tm = import_reference()
        metric = tm.classification.MulticlassConfusionMatrix(num_classes=N_CLASSES, validate_args=False).to(dev)
        update, kind = metric.update, f"the unmodified reference (baseline/_ref, TorchMetrics {tm.__version__}) on CUDA tensors"
    else:
        from oracle.torch_cpu_chain import multiclass_confmat_update_cpu  # device-agnostic restatement of the op chain

        confmat = torch.zeros(N_CLASSES, N_CLASSES, dtype=torch.long, device=dev)
        update = lambda lg, tg: multiclass_confmat_update_cpu(confmat, lg, tg, N_CLASSES)  # noqa: E731
        kind = "reference op chain argmax->t*C+p->bincount->+= (oracle/torch_cpu_chain.py) on CUDA tensors"
    n = len(dev_batches)
    for i in range(3):
        update(*dev_batches[i % n])
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        update(*dev_batches[i % n])
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {"value": UNITS_PER_STEP / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "kind": kind,
            "validate_args": False}


# --------------------------------------------------------------------------------------------------------------
# cfg5 leg: MetricCollection([MulticlassF1Score, MulticlassAUROC], C=1000), 4 x [4096, 1000] f32 per rank
# --------------------------------------------------------------------------------------------------------------
def leg_cfg5(dev, rank: int, world: int, reps: int = 5) -> dict:
    from metrics_b200 import MetricCollection
    from metrics_b200.classification import MulticlassAUROC, MulticlassF1Score

    dist = torch.distributed
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    batches = [(torch.randn(4096, 1000, generator=g, device=dev), torch.randint(0, 1000, (4096,), generator=g, device=dev))
               for _ in range(4)]

    def build():
        return MetricCollection([MulticlassF1Score(num_classes=1000, validate_args=False),
                                 MulticlassAUROC(num_classes=1000, validate_args=False)]).to(dev)

    mc = build()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn):
        out = []
        for _ in range(reps):
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize(dev)
            out.append(e0.elapsed_time(e1))
        t = torch.tensor(out, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # per repetition: the slowest rank
        return float(t.min()), float(t.median())

    def updates():
        mc.reset()
        for lg, tg in batches:
            mc.update(lg, tg)

    def compute():
        for m in mc.values(copy_state=False):
            m._computed = None
            if hasattr(m, "_group_cache"):
                m._group_cache.clear()
        return mc.compute()

    updates()
    compute()
    upd_min, upd_med = timed(updates)
    cmp_min, cmp_med = timed(compute)
    res = compute()
    out = {
        "workload": "MetricCollection([MulticlassF1Score, MulticlassAUROC], num_classes=1000), 4 x [4096,1000] f32 logits per rank "
                    "(BASELINE.json configs[4]); compute() = cross-rank sync + evaluation",
        "update_ms_4_batches": upd_min, "update_ms_4_batches_median": upd_med,
        "update_units_per_s": world * 4 * 4096 * 1000 / (upd_min * 1e-3),
        "compute_ms": cmp_min, "compute_ms_median": cmp_med,
        "f1": float(res["MulticlassF1Score"]), "auroc": float(res["MulticlassAUROC"]),
        "sync_bytes_per_rank": 16384 * 1000 * 4 + 16384 * 8 + 4 * 1000 * 8,
    }
    if world > 1:
        # parity 1: the class-sharded exchange against the reference-shaped "gather everything, evaluate all classes" sync
        os.environ["MB200_SHARDED_CURVES"] = "0"
        gathered = compute()
        g_min, _ = timed(compute)
        os.environ["MB200_SHARDED_CURVES"] = "1"
        assert torch.equal(res["MulticlassAUROC"], gathered["MulticlassAUROC"]), "sharded AUROC differs from the gathered one"
        assert torch.equal(res["MulticlassF1Score"], gathered["MulticlassF1Score"])
        out["compute_ms_gather_everything"] = g_min
        out["compute_path"] = "class-sharded exchange (metrics_b200/parallel_curves.py)"
        # parity 2: small ragged case with ties against the numpy oracle evaluated on the UNION of all ranks' samples
        from oracle import curves as oc

        c_small = 37
        data = []
        for r in range(world):
            gg = torch.Generator().manual_seed(4242 + r)
            n_r = 300 + 17 * r
            # scores already in [0, 1] (no normalisation on either side: the oracle and the kernels see the SAME numbers),
            # quantised to 1/64 so that exact ties abound within and across ranks
            pr = (torch.softmax(torch.randn(n_r, c_small, generator=gg) * 2, 1) * 64).round() / 64
            data.append((pr, torch.randint(0, c_small, (n_r,), generator=gg)))
        small = MulticlassAUROC(num_classes=c_small, average=None, validate_args=False).to(dev)
        small.update(data[rank][0].to(dev), data[rank][1].to(dev))
        got = small.compute().cpu().numpy()
        probs = torch.cat([d[0] for d in data]).numpy()
        want = oc.multiclass_auroc_exact(probs, torch.cat([d[1] for d in data]).numpy(), c_small)
        import numpy as np

        assert np.allclose(got, want, rtol=1e-6, atol=1e-7), "sharded AUROC differs from the oracle on the union"
        out["parity"] = "sharded == gathered (bit-exact, C=1000); sharded == oracle on the union (C=37, ragged, ties, 1e-6)"
    else:
        out["compute_path"] = "local"
    return out


# --------------------------------------------------------------------------------------------------------------
# our arm, cfg2
# --------------------------------------------------------------------------------------------------------------
def run_ours(args) -> dict:
    from metrics_b200 import _native
    from metrics_b200.classification import MulticlassConfusionMatrix

    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    distributed = world > 1
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    sampler = ClockSampler(local_rank)  # child process: starts importing NVML while we set up
    if distributed:
        torch.distributed.init_process_group("nccl", device_id=dev)
    dist = torch.distributed

    if args.config != "cfg2":
        from benchmarks import run_configs

        line = run_configs.bench_line(args, dev, rank, world, sampler)
        if distributed:
            dist.destroy_process_group()
        return line if rank == 0 else {}

    # rank-distinct synthetic shards: two are generated on the host (the e2e leg copies them from pinned memory every
    # step), the rest directly on the device with the same recipe (seeded randn -> bf16, uniform int64 labels)
    host = [make_batch(1000 * rank + i) for i in range(min(2, N_ROT))]
    dev_batches = [(lg.to(dev), tg.to(dev)) for lg, tg in host]
    for i in range(len(host), N_ROT):
        g = torch.Generator(device=dev).manual_seed(1000 * rank + i)
        dev_batches.append((torch.randn(N_ROWS, N_CLASSES, generator=g, device=dev).bfloat16(),
                            torch.randint(0, N_CLASSES, (N_ROWS,), generator=g, device=dev)))
    metric = MulticlassConfusionMatrix(num_classes=N_CLASSES, validate_args=False).to(dev)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput (`value`) -------------------------------------------------------------
    pre = max(args.warmup, 3)
    for i in range(pre):
        metric.update(*dev_batches[i % N_ROT])
    metric.compute()  # untimed: brings up the NCCL communicator / first exchange so that it is not billed to the steps
    if distributed:
        dist.barrier()  # ... and the barrier's own first collective
    sampler.wait_ready()
    metric.reset()
    # Untimed spin-up LAST: communicator bring-up and the sampler hand-shake leave the GPU idle for up to a second, and the
    # first 20-step window after such a pause measures 27 us/step on 8 GPUs against 21.9 us for every later one
    # (profiles/r02_diag_scale_8gpu.json).  The spin-up updates stay in the state: they are part of the expectation below.
    uses = [0] * N_ROT  # how often each resident batch has been folded into the state since the reset
    torch.cuda.synchronize(dev)
    t_spin = time.perf_counter()
    with torch.no_grad():
        while time.perf_counter() - t_spin < 0.25:
            for i in range(64):
                metric.update(*dev_batches[i % N_ROT])
                uses[i % N_ROT] += 1
            torch.cuda.synchronize(dev)

    order = [dev_batches[i % N_ROT] for i in range(args.steps)]
    update = metric.update
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = _native.launch_count()
    w0 = time.time()
    ev0.record()
    with torch.no_grad():  # an evaluation loop: `update` then skips its own grad-mode switch
        for lg, tg in order:
            update(lg, tg)
    ev1.record()
    torch.cuda.synchronize(dev)
    w1 = time.time()
    barrier()
    sampler.window("value", w0, w1)
    launches = _native.launch_count() - launches0
    ms_updates = ev0.elapsed_time(ev1)

    # ---- cross-rank sync of the state: compute() timed on its own, every repetition entered from a barrier -------------------
    sync_ms = []
    w0 = time.time()
    for _ in range(7):
        metric._computed = None
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        result = metric.compute()
        s1.record()
        torch.cuda.synchronize(dev)
        sync_ms.append(s0.elapsed_time(s1))
    sampler.window("sync", w0, time.time())

    # ---- exact check of the timed (and synced) result -------------------------------------------------------------------------
    # every rank re-derives what ITS shard must contribute — per-batch confusion matrices, each from ONE isolated, synchronised
    # update, weighted by how often the batch was cycled through; the expectations are combined over ranks by a DIFFERENT path
    # than the one under test (all_gather + local sum instead of the metric's all-reduce)
    expect = torch.zeros(N_CLASSES, N_CLASSES, dtype=torch.long, device=dev)
    last_batch = (args.steps - 1) % N_ROT
    for b in range(N_ROT):
        times_used = uses[b] + len(range(b, args.steps, N_ROT))  # spin-up + the K timed steps
        if times_used == 0:
            continue
        single = MulticlassConfusionMatrix(num_classes=N_CLASSES, validate_args=False, sync_on_compute=False).to(dev)
        single.update(*dev_batches[b])
        torch.cuda.synchronize(dev)
        expect += single.confmat * times_used
        if b == last_batch:
            last_step = single.compute().clone()
    if distributed:
        slab = torch.empty((world, N_CLASSES, N_CLASSES), dtype=torch.long, device=dev)
        dist.all_gather_into_tensor(slab, expect)
        expect = slab.sum(0)
    n_updates = torch.tensor([sum(uses) + args.steps], dtype=torch.long, device=dev)
    if distributed:
        dist.all_reduce(n_updates)  # ranks spin for the same wall time, not the same number of updates
    assert int(result.sum()) == N_ROWS * int(n_updates), "confusion matrix lost samples"
    assert torch.equal(result, expect), "timed + synced confusion matrix differs from the sum of isolated per-batch updates"
    if args.dump_outputs:
        # The timed state also holds the spin-up updates, whose number depends on wall time; what the LAST timed step adds
        # is the confusion matrix of its batch alone (the check above ties these isolated matrices to the timed state), which
        # is the same from run to run.  Over N ranks: the sum of every rank's last step, as compute() would return it.
        if distributed:
            dist.all_reduce(last_step)
        if rank == 0:
            import numpy as np

            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "confmat.npy"), last_step.cpu().numpy().astype(np.float64))

    per_rank_ms = [ms_updates / args.steps]
    if distributed:  # every rank's own window, for the record (the value uses the maximum)
        slab = torch.empty(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(slab, torch.tensor([ms_updates / args.steps], dtype=torch.float64, device=dev))
        per_rank_ms = [round(float(x), 6) for x in slab.tolist()]
    times = torch.tensor([ms_updates] + sync_ms, dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_updates = float(times[0])
    sync_ms = [float(x) for x in times[1:]]
    # The timed region is EXACTLY the K update steps (events on the launching stream, barrier + synchronize on both sides,
    # max over ranks); the per-epoch compute() (cross-rank sync when N > 1) is timed on its own above (`config.sync`).
    value = UNITS_PER_STEP * args.steps * world / (ms_updates * 1e-3)

    kernel_ms = ms_updates / args.steps  # one kernel launch per step, back to back on one stream
    peak, peak_src = measured_peak_gbs()
    achieved = ALGO_BYTES_PER_LAUNCH / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r01_confmat_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None

    # ---- end to end through the public API: pinned host -> device -> update -> flag read-back, compute at the end
    e2e_steps = max(1, min(args.steps, 64))
    pinned = [(lg.pin_memory(), tg.pin_memory()) for lg, tg in host[:2]]
    m2 = MulticlassConfusionMatrix(num_classes=N_CLASSES, validate_args=True).to(dev)
    stage = [(torch.empty_like(dev_batches[0][0]), torch.empty_like(dev_batches[0][1])) for _ in range(2)]
    for i in range(2):
        stage[i][0].copy_(pinned[i][0], non_blocking=True)
        stage[i][1].copy_(pinned[i][1], non_blocking=True)
        m2.update(*stage[i])
    m2.reset()
    barrier()
    # Double-buffered: the copy of step i+1 is enqueued on copy streams before step i's update() blocks on its validation
    # word, so PCIe never idles; every step still pays its full host->device copy and its device->host flag read.
    n_cs = max(1, int(os.environ.get("MB200_BENCH_E2E_STREAMS", "1")))  # the logits copy is split across this many streams
    copy_streams = [torch.cuda.Stream(device=dev) for _ in range(n_cs)]
    ready = [[torch.cuda.Event() for _ in range(n_cs)] for _ in range(2)]
    main = torch.cuda.current_stream(dev)

    def enqueue_copy(slot: int) -> None:
        rows = N_ROWS // n_cs
        for k, cs in enumerate(copy_streams):
            lo, hi = k * rows, (N_ROWS if k == n_cs - 1 else (k + 1) * rows)
            cs.wait_stream(main)  # the slot's previous consumer (two steps ago) has been enqueued on `main`
            with torch.cuda.stream(cs):
                stage[slot][0][lo:hi].copy_(pinned[slot][0][lo:hi], non_blocking=True)
                if k == 0:
                    stage[slot][1].copy_(pinned[slot][1], non_blocking=True)
                ready[slot][k].record(cs)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    enqueue_copy(0)
    for i in range(e2e_steps):
        s = i % 2
        if i + 1 < e2e_steps:
            enqueue_copy((i + 1) % 2)
        for ev in ready[s]:
            main.wait_event(ev)
        m2.update(*stage[s])  # validate_args=True: reads the kernel's 4-byte validation word back every step
    out_host = m2.compute().cpu()  # the metric result leaves the device
    e1.record()
    barrier()
    sampler.window("e2e", w0, time.time())
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if distributed:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = UNITS_PER_STEP * e2e_steps * world / (float(e2e_ms[0]) * 1e-3)
    assert int(out_host.sum()) == N_ROWS * e2e_steps * world
    h2d = N_ROWS * N_CLASSES * 2 + N_ROWS * 8
    d2h = 4 + (N_CLASSES * N_CLASSES * 8) / e2e_steps
    clocks = sampler.stop()

    extras = {}
    if not args.no_extras:
        extras["cfg5"] = leg_cfg5(dev, rank, world)  # collective: every rank runs it (an error here must stay loud)
        extras["aten"] = aten_gpu_cfg2(dev, dev_batches, max(10, min(args.steps, 50)))
        if world == 1:  # the single-GPU BASELINE configs, so that the driver's N=1 line times them too
            from benchmarks import run_configs

            del dev_batches[2:]
            torch.cuda.empty_cache()

            def secondary(name, fn):  # a failing side leg is reported in the line; it never takes the headline down
                try:
                    extras[name] = fn()
                except Exception as err:  # noqa: BLE001
                    extras[name] = {"error": f"{type(err).__name__}: {err}"}

            secondary("cfg3", lambda: dict(run_configs.leg_cfg3(dev), aten_gpu_baseline=run_configs.aten_cfg3(dev)))
            secondary("cfg4", lambda: run_configs.leg_cfg4(dev))

    cfg = {
        "workload": "MulticlassConfusionMatrix(num_classes=1000).update, [65536,1000] bf16 logits + int64 target"
                    " per GPU per step (BASELINE.json configs[1]); the K timed steps are K update() calls; the per-epoch "
                    "compute() (cross-rank sync) is timed on its own in config.sync and its result is checked exactly",
        "units_per_step_per_gpu": UNITS_PER_STEP, "validate_args": False,
        "l2": f"inputs larger than L2: rotating {N_ROT} distinct 131 MB device batches ({N_ROT * 131} MB >> 126 MB L2)",
        "parallelism": f"dp{world} (independent shards, no data-path collective; one int64 all-reduce of the [C,C] state at compute())",
        "pre_warm": "W warm-up steps, NCCL bring-up, then 0.25 s of untimed updates immediately before the timed window",
        "ms_per_step_per_rank": per_rank_ms,
        "sync": {"what": "metric.compute(): all-reduce of the 8 MB int64 [C,C] state + result clone; 7 repetitions, each entered "
                         "from a barrier, device time, max over ranks" if distributed else "metric.compute() on one GPU (no collective)",
                 "compute_ms_min": min(sync_ms), "compute_ms_median": statistics.median(sync_ms), "state_bytes": N_CLASSES * N_CLASSES * 8,
                 "result_check": "exact: == all_gather + sum of per-rank expectations from isolated per-batch updates"},
    }
    for name in ("cfg5", "cfg3", "cfg4"):
        if name in extras:
            cfg[name] = extras[name]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_updates / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": cfg,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "kernel": "rows_vec_kernel<bf16, ConfmatSink>",
                     "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_LAUNCH,
                     "note": "kernel_ms = back-to-back launch period over the K steps (includes the host latency of the first "
                             "launch); consecutive updates are launched with programmatic stream serialization and wait for the "
                             f"previous grid before their first load (MB200_ROWS_OVERLAP={os.environ.get('MB200_ROWS_OVERLAP', '1')}). "
                             "The peak is a read+write copy; a read-only stream can exceed it."},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "validate_args": True},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if "aten" in extras:
        line["aten_gpu_baseline"] = extras["aten"]
        line["aten_gpu_baseline"]["speedup_device_resident"] = value / world / extras["aten"]["value"]
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        logits0, target0 = make_batch(0)
        n_cpu = 60
        r = time_cpu_chain(logits0, target0, N_ROWS, n_cpu, 3)
        line["cpu_baseline"] = {
            "value": UNITS_PER_STEP / r["median_s"], "unit": UNIT, "cores": r["threads"], "kind": r["kind"],
            "sample": f"{n_cpu} update() calls of the full seed-0 [65536,1000] bf16 batch: {r['what']}, {r['total_s']:.1f} s "
                      f"(per step min {r['min_s'] * 1e3:.2f} ms, median {r['median_s'] * 1e3:.2f} ms)",
        }
    if distributed:
        dist.destroy_process_group()
    return line if rank == 0 else {}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg5 leg and the ATen-on-GPU arm of the cfg2 line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the [C, C] confusion matrix of the last timed step as DIR/confmat.npy (float64; cfg2, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "cfg2"):
        ap.error("--dump-outputs covers the cfg2 line of --impl ours")
    # stdout carries exactly ONE JSON line: everything else that writes to file descriptor 1 (NCCL's version banner with
    # NCCL_DEBUG=VERSION, library chatter) is diverted to stderr; the JSON goes to a private duplicate of the real stdout
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        if int(os.environ.get("RANK", 0)) != 0:
            return
        print(json.dumps(run_reference(args)), file=json_out, flush=True)
        return
    line = run_ours(args)
    if line:
        print(json.dumps(line), file=json_out, flush=True)


if __name__ == "__main__":
    main()
