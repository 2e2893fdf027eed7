#!/usr/bin/env python
"""bench.py — samples/s of PERSIA's sparse-embedding hot path on B200 (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of synthetic Criteo-shaped ids: training forward
(prefix -> per-slot dedup -> find-or-admit over the distinct signs -> gather+pool -> f16) and backward (NaN rule ->
in-order gradient reduce per sign -> Adagrad update).

BASELINE.json names two things, measured by two legs:
  * metric leg — "samples/sec (26 slots, dim128) at 1/2/4/8 B200": dim 128, 8192 samples per GPU (configs[3]'s
    65536 / 8), 1e8 resident rows per GPU, Adagrad.  This is `value` / `e2e` at every N (weak scaling: per-GPU work is
    fixed).  At N >= 2 the rows are hash-sharded over the GPUs and the exchange runs inside the kernels (configs[2]); at
    N = 8 the ids are drawn from a 1e10 key space over a capacity-bounded table with eviction on (configs[3]).
  * roofline leg — configs[1], "1xB200: 26 slots, 1e8 rows, dim-64, batch 4096, GPU hash lookup + sparse Adagrad,
    HBM GB/s vs roofline": run at N = 1 only; `roofline` comes from it.

  python bench.py [--gpus N --steps K --warmup W]            our arm (CUDA, through the C ABI)
  python bench.py --impl reference [...]                     the reference's CPU path (oracle port) on host cores
  python bench.py --dump-outputs DIR [...]                   also write the last timed step's outputs to DIR/*.npy

Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for every field.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from persia_b200 import workload as W  # noqa: E402

METRIC = "samples/sec (Criteo-1TB-shape DLRM sparse path, 26 slots, dim128)"
UNIT = "samples/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=float, default=float(os.environ.get("PB_BENCH_ROWS", 1e8)),
                    help="resident rows per GPU (weak scaling: the table grows with N)")
    ap.add_argument("--batch", type=int, default=8192, help="samples per GPU per step (metric leg)")
    ap.add_argument("--dim", type=int, default=128, help="embedding dim of the metric leg")
    ap.add_argument("--slots", type=int, default=26)
    ap.add_argument("--alpha", type=float, default=1.05)
    ap.add_argument("--keyspace", type=float, default=None,
                    help="key space per GPU the ids are drawn from; default = --rows (everything resident) except at "
                         "N = 8: 1.25e9 per GPU = configs[3]'s 1e10, over a table bounded at --rows with eviction on")
    ap.add_argument("--sets", type=int, default=8, help="rotating input/grad/output buffer sets (> L2 in total)")
    ap.add_argument("--cpu-seconds", type=float, default=float(os.environ.get("PB_BENCH_CPU_SECONDS", 12)))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline-leg", action="store_true", help="N = 1: skip the configs[1] (dim 64) leg")
    ap.add_argument("--no-model-leg", action="store_true", help="N = 1: skip the TrainCtx + DLRM tower leg (e2e_model)")
    ap.add_argument("--no-parity", action="store_true", help="skip the replay of captured steps against the oracle")
    ap.add_argument("--no-staleness", action="store_true", help="skip the 2 / 4 batches-in-flight measurement")
    ap.add_argument("--no-kernel-table", action="store_true", help="N > 1: skip the per-kernel-family timing pass")
    ap.add_argument("--no-graph", action="store_true", help="launch kernel by kernel instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the metric leg's last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "b200" or args.gpus != 1 or args.steps < 1):
        ap.error("--dump-outputs needs --impl b200, --gpus 1 and --steps >= 1")
    return args


def keyspace_per_gpu(args):
    if args.keyspace is not None:
        return float(args.keyspace)
    return 1.25e9 if args.gpus == 8 else float(args.rows)


def workload_config(args):
    """The same dict in both arms (the driver compares them)."""
    n, ks = args.gpus, keyspace_per_gpu(args)
    bounded = ks > args.rows
    which = "configs[3]" if (n == 8 and bounded) else ("configs[2]" if n >= 2 else "configs[2] shape on one GPU")
    return {
        "workload": f"{which}: {args.slots} Criteo-shaped slots, dim {args.dim}, batch {args.batch}/GPU x {n} GPU, "
                    f"{int(args.rows):.3g} resident rows/GPU, key space {ks * n:.3g}"
                    f"{' (capacity-bounded table, eviction on)' if bounded else ''}, Adagrad, training forward + backward",
        "global_batch": args.batch * n, "slots": args.slots, "dim": args.dim, "rows_per_gpu": int(args.rows),
        "key_space_total": int(ks * n), "zipf_alpha": args.alpha, "optimizer": "adagrad(lr=0.01, init=0.01, eps=1e-10)",
        "parallelism": "single shard" if n == 1 else f"rows hash-sharded over {n} GPUs (farmhash64 % {n}), data-parallel "
                                                      f"batches, distinct signs / rows / reduced gradients stored into the "
                                                      f"peer's memory over NVLink by the compute kernels",
    }


# ------------------------------------------------------------------------------------------------------
# clocks: nvidia-smi sampled DURING the timed region (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu_index = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu_index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.2] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, name in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# the reference's CPU path (oracle port): timed on the host cores
# ------------------------------------------------------------------------------------------------------
def host_cores():
    """Cores this process may really use: the affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(p)
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


class CpuArm:
    """The reference's CPU path (oracle port of its EW + PS, in process) on the same workload: a pool of distinct
    batches, admitted once untimed (steady state is a warm table; the GPU arm is timed on a resident table too)."""

    def __init__(self, args, n_threads=None):
        import oracle

        self.S, self.B, self.dim = args.slots, args.batch, args.dim
        self.cores, self.quota = host_cores()
        self.n_threads = n_threads or self.cores
        card = W.scaled_cardinalities(int(keyspace_per_gpu(args) * args.gpus), self.S)
        pf = W.index_prefixes(self.S)
        self.w = oracle.Worker([oracle.SlotCfg(self.dim, prefix=p) for p in pf], n_ps=1, capacity_per_ps=1 << 40,
                               n_internal_shards=max(64, 8 * self.n_threads))
        self.w.configure()
        self.w.set_optimizer(oracle.Optim(oracle.ADAGRAD, lr=0.01, init_acc=0.01, eps=1e-10))
        self.row_off = np.arange(self.S * self.B + 1, dtype=np.uint32)
        rng = np.random.default_rng(123)
        self.g = [(rng.standard_normal((self.B, self.dim)) * 1e-2).astype(np.float16) for _ in range(self.S)]
        self.n_pool = int(min(128, max(2 * self.n_threads, 8)))
        self.ids = W.make_batches(1001, card, self.B, self.n_pool, args.alpha)
        self.warm_seconds = self.run(self.ids)
        self.cursor = 0

    def run(self, ids):
        return self.w.bench(ids, self.row_off, self.B, self.g, self.n_threads)

    def step(self, n_batches):
        """fwd+bwd of the next n_batches of the pool (wraps around); returns seconds."""
        idx = [(self.cursor + i) % self.n_pool for i in range(n_batches)]
        self.cursor = (self.cursor + n_batches) % self.n_pool
        return self.run(np.ascontiguousarray(self.ids[idx]))

    def describe(self, n_batches, reps):
        return (f"median of {reps} repetitions of {n_batches} batches ({self.n_pool} distinct, table warmed by one untimed "
                f"pass) x {self.B} samples x {self.S} slots dim {self.dim}, Adagrad, fwd+bwd, {self.n_threads} threads each "
                f"owning whole batches (in-process EW+PS, no RPC/codec/H2D); affinity+cgroup give {self.cores} cores"
                f"{'' if not self.quota else ' (cpu.max quota %.1f)' % self.quota}")


def cpu_arm(args, seconds):
    arm = CpuArm(args)
    t = arm.step(arm.n_pool)
    per_rep = int(max(arm.n_threads, min(arm.n_pool, arm.n_pool * (seconds / 3.0) / max(t, 1e-3))))
    vals = []
    for _ in range(3):
        tt = arm.step(per_rep)
        vals.append(per_rep * arm.B / tt)
    return {"value": float(np.median(vals)), "unit": UNIT, "cores": arm.n_threads, "kind": "port",
            "sample": arm.describe(per_rep, 3), "spread": [float(min(vals)), float(max(vals))]}


def reference_main(args):
    """--impl reference: the reference's own CPU implementation of the path (no Rust toolchain here, so the
    oracle port) with all the host threads this process may use.  A step = two batches per host thread, fwd+bwd."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args)
    per_step = min(arm.n_pool, 2 * arm.n_threads)
    for _ in range(max(args.warmup, 1)):
        arm.step(per_step)
        if arm.warm_seconds > 20:
            break
    K = max(1, args.steps)
    t0 = time.time()
    times = []
    for _ in range(K):
        times.append(arm.step(per_step))
        if time.time() - t0 > 150:  # keep the whole run within a few minutes
            break
    done = len(times)
    v = done * per_step * arm.B / sum(times)
    line = {
        "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": done, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(times) / done, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "impl": "reference",
        "config": workload_config(args),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": arm.n_threads, "kind": "port",
                         "sample": arm.describe(per_step, done),
                         "median_step_value": float(per_step * arm.B / np.median(times))},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def b200_main(args):
    import torch

    from persia_b200 import native as N

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback; use --impl reference for the CPU arm)"
    if world != args.gpus:
        assert world == 1 and args.gpus == 1, f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})"
    torch.cuda.set_device(local_rank)
    N.load()
    if world > 1:
        import bench_dist

        return bench_dist.run(args, rank, local_rank, world, sys.modules[__name__])
    return single_gpu(args, torch)


def peak_hbm():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    return peak, ("MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)")


def fill_table(torch, SH, sh, card, pf, dev, dim, owner=None):
    """Make the rows of ids [0, card[s]) of every slot resident (the reference's "warm table")."""
    chunk = 1 << 21
    buf = torch.empty((chunk, dim), dtype=torch.float32, device=dev)
    for s in range(len(card)):
        for lo in range(0, int(card[s]), chunk):
            hi = min(int(card[s]), lo + chunk)
            ids = torch.arange(lo, hi, dtype=torch.int64, device=dev)
            signs = SH.add_prefix(ids, [0, hi - lo], [pf[s]])
            if owner is not None:
                signs = signs[SH.shard_of(signs, owner[1]) == owner[0]].contiguous()
            if signs.numel():
                sh.lookup(signs, training=True, out=buf[: signs.numel()])
    torch.cuda.synchronize()
    del buf


def kernel_bytes(stats, dim, state):
    """Algorithmic bytes per launch from the batch's MEASURED multiplicities (SURVEY §8d, with U as observed):
    N id occurrences, U distinct (slot, sign) pairs of which `cold` occur once and `hot` more than 32 times."""
    n, u = stats["occurrences"], stats["items"]
    cold, warm, hot, seg = stats["cold"], stats["warm"], stats["hot"], stats["repeated_occurrences"]
    row = 4 * (dim + state)
    # occurrence lists hold the warm items' occurrences (hot items are filed in the bitmap pool, which is sized to hold
    # every one of them): warm occurrences = list entries, hot occurrences = the rest
    warm_occ = seg
    hot_occ = max(0, n - cold - seg) if hot else 0
    return {
        "k_dedup": n * (8 + 4) + u * 8,                          # ids in, set cell out, distinct list
        "k_probe_items": u * 16,                                 # one index cell per distinct sign
        "k_gather_items": u * 4 * dim + n * 2 * dim,             # each distinct row once + f16 outputs
        "k_nan_scan": n * 2 * dim,
        "k_reduce_cold": cold * (8 + 2 * row + 2 * dim),
        "k_reduce_warm": warm * (16 + 2 * row) + warm_occ * (4 + 2 * dim),
        "k_reduce_hot": hot * (16 + 2 * row) + hot_occ * 2 * dim + hot * 0,
        "worst_case_backward": n * (2 * dim + 16 + 2 * row),
        "whole_step": n * (20 + 2 * dim + 2 * dim) + u * (16 + 4 * dim + 16 + 2 * row),
        "whole_step_worst_case": n * W.algorithmic_bytes_per_id(dim, state, "total"),
    }


DUMP_BYTES = 48 << 20  # what --dump-outputs writes at most: 1260 of the 8192 samples at the default shape


def dump_outputs(out_dir, torch, SH, sh, out, ids, slot_off, pf, B):
    """Writes what one training step gave its caller, for a fixed, seeded sample of the batch's samples (the same
    sample in every slot): `embeddings` [S, n, dim], the pooled f16 embeddings forward returned, as f32; `updated_rows`
    [S, n, dim + optimizer state], the table entries of those samples' signs after backward applied the step's
    gradients; `sample_index` [n], the samples drawn.  Two builds given the same arguments can be compared file for
    file: the inputs are generated from fixed seeds."""
    S = len(pf)
    n = max(1, min(B, DUMP_BYTES // (4 * S * (out.shape[2] + sh.entry_len))))
    idx = np.sort(np.random.default_rng(0).choice(B, size=n, replace=False))
    d_idx = torch.from_numpy(idx).to(out.device)
    signs = SH.add_prefix(ids, slot_off, pf).view(S, B).index_select(1, d_idx).reshape(-1)
    rows, found = sh.get_entries(signs)
    assert bool(found.all()), "a sign the step just updated is not in the table"
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"embeddings": out.index_select(1, d_idx).float(), "updated_rows": rows.view(S, idx.size, -1),
              "sample_index": torch.from_numpy(idx.astype(np.float64))}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def run_leg(args, torch, dim, B, rows, name, want_kernels, want_parity, dump_dir=None):
    """One single-GPU leg: table of `rows` resident rows of `dim`, batches of B samples."""
    import ctypes as C

    from persia_b200 import native as N
    from persia_b200 import shard as SH

    lib = N.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    S, K, Wm = args.slots, args.steps, max(args.warmup, 3)
    card = W.scaled_cardinalities(rows, S)
    pf = W.index_prefixes(S)
    slot_off = [s * B for s in range(S + 1)]
    n_occ = S * B
    sh = SH.EmbeddingShard(dim, rows + 1024, dev)
    sh.set_optimizer(N.OPT_ADAGRAD, lr=0.01, initialization=0.01, eps=1e-10)
    sh.configure()
    ctx = SH.BatchContext(n_occ, n_occ, pf, device=dev)
    t_fill = time.time()
    fill_table(torch, SH, sh, card, pf, dev, dim)
    resident = len(sh)
    t_fill = time.time() - t_fill
    assert resident == rows, (resident, rows)

    # ---- rotating buffer sets: ids, gradients, outputs (together > L2) ; pinned host ids for e2e
    n_sets = max(2, args.sets)
    n_sets += n_sets % 2  # (the e2e staging buffers alternate with the sets)
    ids_host = W.make_batches(2, card, B, n_sets, args.alpha)
    ids_pinned = torch.from_numpy(ids_host.view(np.int64)).pin_memory()
    ids_dev = [ids_pinned[k].to(dev) for k in range(n_sets)]
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    grads_all = (torch.randn((n_sets, S, B, dim), generator=g, device=dev) * 1e-2).half()
    grads = [[grads_all[k, s] for s in range(S)] for k in range(n_sets)]
    outs = [torch.empty((S, B, dim), dtype=torch.float16, device=dev) for _ in range(n_sets)]

    def step(k):
        ctx.forward(sh, ids_dev[k], slot_off, B, training=True, out=outs[k])
        ctx.backward(sh, grads[k])

    res = {"name": name, "dim": dim, "batch": B}
    stream = torch.cuda.Stream(device=dev)
    use_graph = not args.no_graph
    with torch.cuda.stream(stream):
        for i in range(3):
            step(i % n_sets)
        stream.synchronize()
        l0 = lib.pb_launch_count()
        step(0)
        launches_per_step = int(lib.pb_launch_count() - l0)
        stream.synchronize()
        stats = ctx.batch_stats()
        graphs = None
        if use_graph:
            graphs = []
            for k in range(n_sets):
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=stream):
                    step(k)
                graphs.append(gph)

        def run(i):
            if graphs is not None:
                graphs[i % n_sets].replay()
            else:
                step(i % n_sets)

        for i in range(Wm):
            run(i)
        stream.synchronize()
        sampler = ClockSampler(dev.index or 0)
        sampler.start()
        time.sleep(0.25)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.time()
        e0.record(stream)
        for i in range(K):
            run(i)
        e1.record(stream)
        torch.cuda.synchronize()
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop(t0, t1)
        if dump_dir is not None:  # before the passes below overwrite the output buffers and update the table again
            k = (K - 1) % n_sets
            dump_outputs(dump_dir, torch, SH, sh, outs[k], ids_dev[k], slot_off, pf, B)
        reps = []
        for _ in range(3):  # run-to-run spread of the same K steps
            e0.record(stream)
            for i in range(K):
                run(i)
            e1.record(stream)
            torch.cuda.synchronize()
            reps.append(e0.elapsed_time(e1) / K)

        kern = None
        if want_kernels:
            # per-kernel durations: CUDA events around every launch of ONE family at a time on its launching stream
            # (bracketing all launches at once makes the host the bottleneck and small kernels read high)
            fam_names = ["k_probe_items", "k_dedup", "k_gather_items", "k_nan_scan", "k_reduce_hot", "k_reduce_cold", "other",
                         "k_reduce_warm"]
            n_prof = min(K, 40)
            kern = {}
            for f in (0, 1, 2, 3, 4, 5, 7):
                lib.pb_profile_enable(1 << f)
                for i in range(n_prof):
                    step(i % n_sets)
                fam_ms = (C.c_double * 8)()
                fam_cnt = (C.c_uint64 * 8)()
                N.check(lib.pb_profile_read(fam_ms, fam_cnt, 8))
                lib.pb_profile_enable(0)
                if fam_cnt[f]:
                    kern[fam_names[f]] = {"us": 1e3 * fam_ms[f] / fam_cnt[f], "launches_per_step": fam_cnt[f] / n_prof}

        # ---- e2e: host ids (pinned) -> H2D -> forward -> backward -> D2H of the per-slot status, every step, a host sync
        # per step (the caller reads every step's status, one step behind the launches).  The ids of step i + 1 are copied on a copy
        # stream while step i computes (the reference's Forward engine prefetches batches the same way, forward.rs:470-
        # 780); every copy is inside the timed region.
        status_host = [torch.empty(S, dtype=torch.int32).pin_memory() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        ids_stage = [torch.empty(n_occ, dtype=torch.int64, device=dev) for _ in range(2)]
        out_e2e = outs[0]
        copy_stream = torch.cuda.Stream(device=dev)
        ev_copied = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]

        def e2e_compute(k):
            ctx.forward(sh, ids_stage[k % 2], slot_off, B, training=True, out=out_e2e)
            st = ctx.backward(sh, grads[k], want_status=True)
            status_host[k % 2].copy_(st, non_blocking=True)

        def e2e_copy(k):  # enqueue the H2D of set k into its staging buffer once the step that last used it is done
            b = k % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_free[b])
                ids_stage[b].copy_(ids_pinned[k], non_blocking=True)
                ev_copied[b].record(copy_stream)

        e2e_graphs = None
        if use_graph:  # forward + backward + the status D2H of a step are one graph per buffer set
            for b in range(2):
                ids_stage[b].copy_(ids_pinned[b])
            e2e_compute(0)
            stream.synchronize()
            e2e_graphs = []
            for k in range(n_sets):
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=stream):
                    e2e_compute(k)
                e2e_graphs.append(gph)
        for b in range(2):
            ev_free[b].record(stream)
        stream.synchronize()

        seen = [0]

        def e2e_run(n):
            e2e_copy(0)
            for i in range(n):
                k = i % n_sets
                e2e_copy((i + 1) % n_sets)  # the next step's ids travel while this step computes
                stream.wait_event(ev_copied[k % 2])
                if e2e_graphs is not None:
                    e2e_graphs[k].replay()
                else:
                    e2e_compute(k)
                ev_free[k % 2].record(stream)
                ev_done[k % 2].record(stream)
                if i:  # the host reads every step's status, one step behind the launches (two pinned result buffers)
                    ev_done[(k - 1) % 2].synchronize()
                    seen[0] += int(status_host[(k - 1) % 2][0] >= 0)
            ev_done[(n - 1) % n_sets % 2].synchronize()
            seen[0] += int(status_host[(n - 1) % n_sets % 2][0] >= 0)
            copy_stream.synchronize()

        assert n_sets % 2 == 0, "the staging buffers alternate with the buffer sets"
        e2e_run(Wm)
        torch.cuda.synchronize()
        e0.record(stream)
        e2e_run(K)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_e2e = e0.elapsed_time(e1)

        parity = None
        if want_parity:
            parity = parity_single(torch, sh, run, outs, ids_host, grads_all, pf, S, B, dim, dev, stream)

    # ---- embedding_staleness > 1 (persia/ctx.py:1021-1040: that many batches between lookup and update): J batches in
    # flight, each with its own context, stream and graphs.  Not the parity configuration (the reference is not
    # deterministic there either); reported beside `value`, which stays at staleness 1.
    in_flight = {}
    if use_graph and not args.no_staleness:
        for J in (2, 4):
            if n_sets < J:
                break
            ctxs = [SH.BatchContext(n_occ, n_occ, pf, device=dev) for _ in range(J)]
            streams = [torch.cuda.Stream(device=dev) for _ in range(J)]
            gs = [[None] * n_sets for _ in range(J)]
            for j in range(J):
                with torch.cuda.stream(streams[j]):
                    for k in range(j, n_sets, J):
                        ctxs[j].forward(sh, ids_dev[k], slot_off, B, training=True, out=outs[k])
                        ctxs[j].backward(sh, grads[k])
                        streams[j].synchronize()
                        gph = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gph, stream=streams[j]):
                            ctxs[j].forward(sh, ids_dev[k], slot_off, B, training=True, out=outs[k])
                            ctxs[j].backward(sh, grads[k])
                        gs[j][k] = gph
            torch.cuda.synchronize()

            def fly(n):
                for i in range(n):
                    k = i % n_sets
                    j = k % J
                    with torch.cuda.stream(streams[j]):
                        gs[j][k].replay()

            fly(Wm)
            torch.cuda.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            done = [torch.cuda.Event() for _ in range(J)]
            ev[0].record(streams[0])
            for j in range(1, J):
                streams[j].wait_event(ev[0])
            fly(K)
            for j in range(1, J):
                done[j].record(streams[j])
                streams[0].wait_event(done[j])
            ev[1].record(streams[0])
            torch.cuda.synchronize()
            in_flight[str(J)] = {"ms_per_step": ev[0].elapsed_time(ev[1]) / K,
                                 "samples_per_s": B * K / (ev[0].elapsed_time(ev[1]) * 1e-3)}
            del gs
            for c in ctxs:
                c.close()
    wait_errors = sh.counters()["wait_errors"]
    assert wait_errors == 0, "an in-kernel wait gave up: the run is void"
    res.update(ms_per_step=ms / K, ms_per_step_reps=reps, ms_e2e=ms_e2e / K, launches_per_step=launches_per_step,
               stats=stats, kernels=kern, clocks=clocks, resident=resident, t_fill=round(t_fill, 2), parity=parity,
               n_sets=n_sets, graph=graphs is not None, in_flight=in_flight,
               l2="inputs larger than L2: %.1f GB table + %d rotating id/grad/output sets (%.0f MB)" % (
                   resident * 4.0 * 2 * dim / 1e9, n_sets, n_sets * 2 * n_occ * dim * 2 / 1e6))
    del graphs, e2e_graphs
    ctx.close()
    sh.close()
    del grads_all, grads, outs, ids_dev
    torch.cuda.empty_cache()
    return res


def parity_single(torch, sh, run, outs, ids_host, grads_all, pf, S, B, dim, dev, stream):
    """Replays two of the timed (graph-captured) steps from the table's current state and checks outputs and every
    touched row against the oracle, bit for bit (Adagrad in the oracle's exact-rsqrt mode).  The oracle is the checker
    here, never the thing measured."""
    import oracle

    sets = (0, 1)
    signs = np.unique(np.concatenate([oracle.add_prefix(ids_host[k][i * B:(i + 1) * B], 8, pf[i]) for k in sets for i in range(S)]))
    d_signs = torch.from_numpy(signs.view(np.int64)).to(dev)
    ent, found = sh.get_entries(d_signs)
    assert bool(found.all())
    w = oracle.Worker([oracle.SlotCfg(dim, prefix=p) for p in pf], n_ps=1, capacity_per_ps=1 << 40)
    w.configure()
    w.set_optimizer(oracle.Optim(oracle.ADAGRAD, lr=0.01, init_acc=0.01, eps=1e-10))
    w.set_embedding(signs, ent.cpu().numpy(), dim)
    oracle.set_rsqrt_exact(True)
    try:
        row_off = np.arange(S * B + 1, dtype=np.uint32)
        for k in sets:
            run(k)
            stream.synchronize()
            want, octx = w.forward(ids_host[k], row_off, B, training=True)
            got = outs[k].cpu().numpy()
            for i in range(S):
                if got[i].tobytes() != want[i].tobytes():
                    raise AssertionError(f"parity: forward output of slot {i} differs from the oracle")
            gk = grads_all[k].cpu().numpy()
            w.backward(octx, [gk[i] for i in range(S)])
        ent2 = sh.get_entries(d_signs)[0].cpu().numpy()
        bad = sum(ent2[j].tobytes() != w.get_entry(int(s)).tobytes() for j, s in enumerate(signs))
        if bad:
            raise AssertionError(f"parity: {bad} of {signs.size} updated rows differ from the oracle")
    finally:
        oracle.set_rsqrt_exact(False)
    return {"checked": True, "steps_replayed": len(sets), "rows_compared": int(signs.size),
            "what": "graph-captured steps replayed from the live table; outputs and rows bit-identical to the oracle"}


def roofline_from(leg, peak, peak_src, label):
    dim, B = leg["dim"], leg["batch"]
    st = leg["stats"]
    by = kernel_bytes(st, dim, dim)
    kern = leg["kernels"] or {}
    table = {}
    for k, v in kern.items():
        if k in by:
            gbs = by[k] / (v["us"] * 1e-6) / 1e9
            table[k] = {"us": round(v["us"], 2), "algorithmic_bytes": int(by[k]), "achieved_gbs": round(gbs, 1),
                        "frac": round(gbs / peak, 4)}
    dom = "k_reduce_cold"  # the kernel that moves the most bytes: row in, row out, gradient in, for every sign seen once
    ach = table.get(dom, {}).get("achieved_gbs")
    step_s = leg["ms_per_step"] * 1e-3
    hot_max = max(1, st.get("max_multiplicity", 0))
    return {
        "bound": "hbm", "kernel": "k_reduce_cold (A8+A9 of the signs occurring once in the batch — most distinct signs: gradient "
                                  "prepared, Adagrad step + weight bound on the resident row) on " + label,
        "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if ach else None,
        "frac_worst_case": by["whole_step_worst_case"] / step_s / 1e9 / peak,
        "traffic": None,
        "traffic_note": "not measured by this run: profiles/ holds the ncu --set full capture of this command "
                        "(dram__bytes_read.sum + dram__bytes_write.sum per kernel) and its command line",
        "peak_source": peak_src,
        "bytes_model": "measured multiplicities of the batch: N occurrences, U distinct (slot, sign) pairs, of which `cold` occur "
                       "once, `warm` 2..32 times (their occurrences are counted), `hot` more.  k_reduce_cold = cold x (8 + "
                       "8(D+S) + 2D); k_reduce_warm = warm x (16 + 8(D+S)) + their occurrences x (4 + 2D); k_reduce_hot = hot x "
                       "(16 + 8(D+S)) + their occurrences x 2D.  frac_worst_case: the whole step's U = N bytes (SURVEY 8d) over "
                       "the measured step time.  k_reduce_hot is not bandwidth-bound: the reference's summation order makes a "
                       "sign's occurrences one dependent f32 add after another (its floor is the largest multiplicity x ~7 cycles)",
        "unique_fraction": st["items"] / max(1, st["occurrences"]), "batch_stats": st,
        "kernels": table,
        "whole_step": {"ms": leg["ms_per_step"], "samples_per_s": B / step_s,
                       "algorithmic_bytes": int(by["whole_step"]), "achieved_gbs": by["whole_step"] / step_s / 1e9,
                       "frac": by["whole_step"] / step_s / 1e9 / peak,
                       "frac_worst_case": by["whole_step_worst_case"] / step_s / 1e9 / peak},
    }


def model_leg(args, torch, steps, warmup):
    """e2e_model: the same sparse path driven the way a user drives it — persia_b200.api.TrainCtx (the persia.ctx API)
    with a DLRM-style PyTorch dense tower: host numpy batch -> PersiaBatch -> get_embedding_from_data -> model forward
    -> BCE loss -> ctx.backward (dense SGD step + sparse Adagrad update), every step, wall clock around the loop."""
    from persia_b200 import api
    from persia_b200 import persia_core as PC

    S, B, dim, n_dense = args.slots, args.batch, args.dim, 13
    names = [f"C{i + 1}" for i in range(S)]
    PC.reset()
    PC._S.capacity = int(min(args.rows, 2e7)) + 1024
    PC.set_embedding_config({"slots_config": {n: {"dim": dim} for n in names}})
    card = W.scaled_cardinalities(int(min(args.rows, 2e7)), S)
    torch.manual_seed(0)
    prev_precision = torch.get_float32_matmul_precision()
    torch.set_float32_matmul_precision("high")  # the dense tower's GEMMs on the tensor cores (TF32); the sparse path is untouched
    model = W.make_dlrm_tower(S, dim, n_dense=n_dense).cuda()
    dense_opt = torch.optim.SGD(model.parameters(), lr=0.01)
    loss_fn = torch.nn.BCEWithLogitsLoss()
    n_pool = 8
    ids_pool = W.make_batches(7, card, B, n_pool, args.alpha).reshape(n_pool, S, B)
    rng = np.random.default_rng(11)
    dense_pool = rng.standard_normal((n_pool, B, n_dense)).astype(np.float32)
    label_pool = (rng.random((n_pool, B, 1)) < 0.25).astype(np.float32)
    losses = []
    with api.TrainCtx(model=model, embedding_optimizer=api.Adagrad(lr=0.01, initial_accumulator_value=0.01, eps=1e-10),
                      dense_optimizer=dense_opt, device_id=torch.cuda.current_device(), mixed_precision=False) as ctx:
        def step(k):
            pb = api.PersiaBatch([api.IDTypeFeatureWithSingleID(names[i], ids_pool[k, i]) for i in range(S)],
                                 non_id_type_features=[api.NonIDTypeFeature(dense_pool[k], name="dense")],
                                 labels=[api.Label(label_pool[k], name="click")], requires_grad=True)
            tb = ctx.get_embedding_from_data(pb)
            out, labels = ctx.forward(tb)
            loss = loss_fn(out, labels[0].squeeze(1))
            ctx.backward(loss)
            return loss

        for i in range(warmup):
            step(i % n_pool)
        torch.cuda.synchronize()
        t0 = time.time()
        for i in range(steps):
            losses.append(step(i % n_pool))
        ctx.backward_engine.flush()
        torch.cuda.synchronize()
        dt = time.time() - t0
    res = {"value": B * steps / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / steps, "steps": steps,
           "first_loss": float(losses[0]), "last_loss": float(losses[-1]),
           "path": f"numpy batch -> api.PersiaBatch -> TrainCtx.get_embedding_from_data -> DLRM tower ({sum(p.numel() for p in model.parameters())} "
                   f"dense parameters, fp32 weights, TF32 matmuls) -> BCE -> TrainCtx.backward (dense SGD + sparse Adagrad); {int(min(args.rows, 2e7)):.3g}-id key space, "
                   "rows admitted on the fly", "h2d_bytes_per_step": S * B * 8 + B * n_dense * 4 + B * 4}
    PC.reset()
    torch.set_float32_matmul_precision(prev_precision)
    torch.cuda.empty_cache()
    return res


def single_gpu(args, torch):
    peak, peak_src = peak_hbm()
    rows = int(args.rows)
    roof_leg = None
    if not args.no_roofline_leg:
        roof_leg = run_leg(args, torch, 64, 4096, rows, "roofline leg (configs[1])", True, not args.no_parity)
    leg = run_leg(args, torch, args.dim, args.batch, rows, "metric leg", True, not args.no_parity, args.dump_outputs)
    B, K = args.batch, args.steps
    S = args.slots
    n_occ = S * B
    value = B / (leg["ms_per_step"] * 1e-3)
    metric_roof = roofline_from(leg, peak, peak_src, f"the metric leg: dim {args.dim}, batch {B}, {rows:.3g} rows")
    if roof_leg:
        roofline = roofline_from(roof_leg, peak, peak_src, "configs[1]: dim 64, batch 4096, 1e8 rows")
        roofline["metric_leg"] = {k: metric_roof[k] for k in ("achieved", "frac", "frac_worst_case", "kernels", "whole_step",
                                                              "unique_fraction", "batch_stats")}
    else:
        roofline = metric_roof
    e2e_model = None
    if not args.no_model_leg:
        e2e_model = model_leg(args, torch, steps=min(K, 50), warmup=10)
    cpu = None
    if not args.no_cpu_baseline:
        c = cpu_arm(args, args.cpu_seconds)
        cpu = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample", "spread")}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": max(args.warmup, 3),
        "ms_per_step": leg["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "run": {"ms_per_step_repetitions": leg["ms_per_step_reps"], "resident_rows": leg["resident"],
                "table_fill_seconds": leg["t_fill"], "l2": leg["l2"],
                "launch": ("CUDA graph replay, one graph per buffer set" if leg["graph"] else "kernel by kernel") +
                          "; pb_backward forks the hot-sign reduce onto the context's own stream",
                "reduce_order": "reference order for every multiplicity (bit-exact vs the oracle)",
                "batches_in_flight": {"note": "embedding_staleness 2 / 4: that many batches in flight on their own contexts and "
                                              "streams over the same table; `value` is staleness 1 (the parity configuration)",
                                      **leg["in_flight"],
                                      "roofline_leg": roof_leg["in_flight"] if roof_leg else None},
                "roofline_leg": None if not roof_leg else {
                    "workload": "configs[1]: 26 slots, 1e8 rows, dim 64, batch 4096, Adagrad", "ms_per_step": roof_leg["ms_per_step"],
                    "samples_per_s": 4096 / (roof_leg["ms_per_step"] * 1e-3), "ms_per_step_repetitions": roof_leg["ms_per_step_reps"],
                    "e2e_samples_per_s": 4096 / (roof_leg["ms_e2e"] * 1e-3), "parity": roof_leg["parity"]}},
        "clocks": leg["clocks"],
        "e2e": {"value": B / (leg["ms_e2e"] * 1e-3), "unit": UNIT, "h2d_bytes_per_step": n_occ * 8,
                "d2h_bytes_per_step": S * 4, "ms_per_step": leg["ms_e2e"],
                "path": "pinned host ids -> H2D (copy stream, one step ahead) -> pb_forward -> pb_backward -> D2H slot status read by the host every step, one step behind the launches"},
        "e2e_model": e2e_model,
        "gpu_launches": leg["launches_per_step"] * K,
        "parity_checked": bool(leg["parity"] and leg["parity"]["checked"]), "parity": leg["parity"],
        "roofline": roofline,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_main(args)
    else:
        b200_main(args)


if __name__ == "__main__":
    main()
