#!/usr/bin/env python
"""bench.py -- pan/core permutations per second on B200 (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|c1|c5|c3] [--perms P] [--dump-outputs DIR]
    python bench.py --impl reference ...          # the CPU arm (oracle C port, all host threads)
    torchrun --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU

The library is the one build() (python -m pangenomix_b200.build) left in the tree; bench.py compiles nothing.
--dump-outputs DIR writes what the timed path returned in its last step as DIR/<name>.npy (float64, at most
64 MB in all; rows of a larger output are a fixed seeded sample), so that two builds can be compared on the
same inputs: the table, the permutations and the Bernoulli points are all drawn from fixed seeds.

A step is one pass of the hot path over one batch of permutations: P genome orders
(per GPU) -> P pan/core curves, through libpgx_b200 (include/pgx.h).  The default workload
is config C4 of BASELINE.json (10,000 genomes x 200,000 genes, 10,000 permutations), the
configuration the north_star's roofline and scaling targets are quoted on.

  value : permutations/s, table and permutations resident in HBM, CUDA-event timed,
          max over ranks (weak scaling: every rank rarefies its own P permutations of the
          replicated table; for N > 1 the int32 curves of every step are gathered on rank 0
          inside the timed region -- pushed into rank 0's symmetric-memory buffer over NVLink,
          asynchronously, overlapped with the next step; NCCL gather as fallback).
  e2e   : the same through the host-buffer C-ABI call (pinned host permutations in,
          host curves out; copies inside the timed region).
  roofline : the slower of the two row kernels against the pipe that binds it -- the list kernel against
          the shared-memory / LSU data pipe (wavefronts from the committed ncu capture x 128 B over its live
          CUDA-event duration, a separate pass: the timed region runs the two kernels side by side), the
          probe kernel against instruction issue; SURVEY.md section 8d's HBM bookkeeping (4 nnz + 4 (G + 1)
          algorithmic bytes per permutation, measured HBM copy peak of MEASURED_PEAKS.json, DRAM bytes
          from ncu) is kept under roofline.hbm as an EFFECTIVE fraction.
  cpu_baseline : the oracle's C port of the reference algorithm on a bounded sample.
  api   : the reference-facing Python call itself, estimate_pan_core_size(df, 2000): host RNG
          stream + H2D + kernels + D2H + float64 DataFrame.
  heaps : pgx_heaps_fit on the curves of one step next to scipy curve_fit (SURVEY.md 8f).
  beta_binomial : table marginals + compute_beta_binomial_core_genome with its Monte-Carlo KS on the GPU (8f rank 4).
--workload c3 prints the same kind of line for the Bernoulli grid (LL + gradient evaluations/s,
whole-fit time).  One JSON line on stdout (rank 0); everything else goes to stderr.
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

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

METRIC = "pan_core_permutations_per_sec"
UNIT = "perms/s"
FALLBACK_HBM_GBS = 6650.0        # /opt/skills/guides/B200_PROFILING.md fallback


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c1", "c2", "c4", "c5", "c3"],
                    help="c4/c2/c1/c5: pan/core rarefaction (c4 is the headline metric; c5 = 50,000 genomes x 2,000,000 "
                         "alleles needs minutes of host time to generate and plan); c3: Bernoulli-grid LL+gradient")
    ap.add_argument("--genes", type=int, default=40000, help="c3: genes of the Bernoulli grid (400 genomes)")
    ap.add_argument("--perms", type=int, default=0, help="permutations per GPU per step (0 = the config's)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-check", action="store_true",
                    help="N > 1: rank 0 also runs the cpu_baseline leg (oracle check of its GPU curves) while the others wait")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, what the driver runs): every GPU rarefies the config's permutation count; "
                         "strong: the config's permutations are split over the GPUs, as BASELINE.json words C4")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT = 64_000_000            # bytes --dump-outputs writes at most


def dump_rows(n_rows, row_bytes, reserved):
    """Row indices --dump-outputs keeps of an output of ``n_rows`` rows: all of them when they fit DUMP_LIMIT,
    else a sample fixed by seed 0 (so two runs with the same arguments keep the same rows)."""
    k = min(n_rows, (DUMP_LIMIT - reserved) // (row_bytes + 8))
    if k == n_rows:
        return np.arange(n_rows)
    return np.sort(np.random.RandomState(0).choice(n_rows, k, replace=False))


def dump_outputs(out_dir, arrays):
    """Writes every array of ``arrays`` (float32 or float64) as out_dir/<name>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, arr in arrays.items():
        arr = np.ascontiguousarray(arr)
        assert arr.dtype in (np.float32, np.float64), (name, arr.dtype)
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, arr)
        total += os.path.getsize(path)
    assert total <= DUMP_LIMIT, "dumped %d bytes" % total
    log("[bench] wrote %s (%.1f MB) to %s" % (", ".join(sorted(arrays)), total / 1e6, out_dir))


# --------------------------------------------------------------------------------------
# workload
# --------------------------------------------------------------------------------------
def load_matrix(name, rank, barrier):
    """Synthetic table of SURVEY.md section 8d; generated once per box and cached in /tmp."""
    import scipy.sparse
    from pangenomix_b200 import synth
    n_genes, n_genomes, _, seed, _ = synth.CONFIGS[name]
    cache = os.path.join(tempfile.gettempdir(), "pgx_synth_%s_%d.npy" % (name, seed))
    if rank == 0 and not os.path.exists(cache):
        t = time.time()
        coo = synth.config_matrix(name)
        packed = np.stack([coo.row.astype(np.int32), coo.col.astype(np.int32)])
        tmp = cache + ".tmp%d.npy" % os.getpid()
        np.save(tmp, packed)
        os.replace(tmp, cache)
        log("[bench] generated %s %s nnz=%d in %.1fs" % (name, coo.shape, coo.nnz, time.time() - t))
    barrier()
    packed = np.load(cache)
    data = np.ones(packed.shape[1], dtype=np.int64)
    return scipy.sparse.coo_matrix((data, (packed[0], packed[1])), shape=(n_genes, n_genomes))


def workload_config(name, coo, perms, world, scaling="weak"):
    return {
        "workload": "%s: estimate_pan_core_size on a synthetic %d-genome x %d-gene presence/absence "
                    "table (nnz %d), %d permutations %s per step" % (
                        name.upper(), coo.shape[1], coo.shape[0], coo.nnz, perms,
                        "per GPU" if scaling == "weak" else "split over the GPUs"),
        "n_genomes": int(coo.shape[1]), "n_genes": int(coo.shape[0]), "nnz": int(coo.nnz),
        "perms_per_gpu": int(perms if scaling == "weak" else -(-perms // world)),
        "parallelism": "permutation shards x%d, table replicated" % world,
    }


# --------------------------------------------------------------------------------------
# CPU arm (oracle C port)
# --------------------------------------------------------------------------------------
def cpu_sample(coo, n_genomes, budget_s, threads):
    """Times the C port of pangenome_analysis.py:81-90 on a bounded sample of permutations."""
    from oracle import cport
    gm = cport.GenomeMajor(coo)
    rng = np.random.RandomState(1)
    one = np.stack([rng.permutation(n_genomes)]).astype(np.int32)
    t = time.perf_counter()
    cport.curves_direct(gm, one, n_threads=1)
    t1 = time.perf_counter() - t
    per_thread = max(1, int(round(budget_s / max(t1, 1e-6))))
    sample = threads * per_thread
    perms = np.stack([rng.permutation(n_genomes) for _ in range(sample)]).astype(np.int32)
    return gm, perms, t1


def python_reference_sample(coo, eng=None, n_iter=1):
    """The UNMODIFIED Python reference (vendored into git-ignored baseline/_ref by baseline/vendor_ref.py) on
    ``n_iter`` permutations of the same table: its own estimate_pan_core_size, one host core as the reference runs.
    With an engine, the GPU curves of the same seed are checked against the reference's output bit for bit."""
    try:
        from baseline import vendor_ref
        ref_pa, ref_su = vendor_ref.import_reference()
    except ImportError as exc:
        return {"unavailable": str(exc)}
    import contextlib
    import io
    from pangenomix_b200 import synth
    index, columns = synth.labels_for(*coo.shape)
    lsdf = ref_su.LightSparseDataFrame(index, columns, coo)
    np.random.seed(12345)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        df = ref_pa.estimate_pan_core_size(lsdf, n_iter)
    dt = time.perf_counter() - t0
    out = {"value": n_iter / dt, "unit": UNIT, "cores": 1, "kind": "reference", "seconds": dt,
           "sample": "%d permutation(s) of the same table through the reference's own estimate_pan_core_size "
                     "(pangenome_analysis.py:51-98, numpy %s), incl. its COO -> CSR conversion" % (n_iter, np.__version__)}
    if eng is not None:
        from pangenomix_b200 import engine
        np.random.seed(12345)
        perms = engine.draw_legacy_permutations(coo.shape[1], n_iter)
        out["gpu_curves_equal_reference"] = bool(np.array_equal(eng.curves_host(perms, out_f64=True), df.values))
        assert out["gpu_curves_equal_reference"], "GPU != Python reference"
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import cport
    from pangenomix_b200 import synth
    coo = load_matrix(args.workload, 0, lambda: None)
    perms_cfg = args.perms or synth.CONFIGS[args.workload][4]
    threads = os.cpu_count() or 1
    gm, perms, t1 = cpu_sample(coo, coo.shape[1], max(1.0, args.cpu_seconds / 4.0), threads)
    for _ in range(args.warmup):
        cport.curves_direct(gm, perms[:threads], n_threads=threads)
    t = time.perf_counter()
    for _ in range(args.steps):
        pan, core = cport.curves_direct(gm, perms, n_threads=threads)
    dt = time.perf_counter() - t
    if args.dump_outputs:
        curves = np.hstack([pan, core])
        rows = dump_rows(curves.shape[0], curves.shape[1] * 8, curves.shape[1] * 8 + 4096)
        dump_outputs(args.dump_outputs, {"curves": curves[rows], "curve_rows": rows.astype(np.float64),
                                         "mean_curve": curves.mean(axis=0)})
    value = perms.shape[0] * args.steps / dt
    sample = "%d permutations per step (of the config's %d), %d threads, oracle C port of " \
             "pangenome_analysis.py:81-90" % (perms.shape[0], perms_cfg, threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic", "config": workload_config(args.workload, coo, perms_cfg, world),
        "cells_per_s": value * coo.shape[0] * coo.shape[1],
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "single_thread_s_per_perm": t1,
                         "reference_python": python_reference_sample(coo, None, n_iter=1 if coo.shape[1] >= 2000 else 20)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ["clocks.sm", "clocks.max.sm", "power.draw",
              "clocks_event_reasons.hw_slowdown", "clocks_event_reasons.hw_thermal_slowdown",
              "clocks_event_reasons.sw_thermal_slowdown", "clocks_event_reasons.sw_power_cap"]

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + ",".join(self.FIELDS),
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        sm, sm_max, power, reasons = [], 0.0, 0.0, set()
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.05:
                continue
            parts = [p.strip() for p in line.split(",")]
            if len(parts) != len(self.FIELDS):
                continue
            try:
                sm.append(float(parts[0]))
                sm_max = max(sm_max, float(parts[1]))
                power = max(power, float(parts[2]))
            except ValueError:
                continue
            for name, flag in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                  parts[3:]):
                if flag == "Active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": sm_max or None,
                "power_w_max": power or None, "samples": len(sm), "reasons": sorted(reasons)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()


def measured_peak():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, KeyError, ValueError):
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_counters(workload, kind):
    """Per-permutation counters of a kernel from the committed ncu capture (profiles/roofline_traffic.json, written
    by scripts/ncu_summary.py from the ``ncu --set full`` report of the same workload): DRAM bytes, LSU wavefronts,
    pipe utilisations.  Empty when nothing is committed for this workload."""
    try:
        with open(os.path.join(REPO, "profiles", "roofline_traffic.json")) as f:
            return dict(json.load(f)[workload][kind])
    except (OSError, ValueError, KeyError, TypeError):
        return {}


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from pangenomix_b200 import _native, engine, synth

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()

    barrier()
    _native.load()
    l2_bytes = int(_native.device_info()["l2_bytes"])
    coo = load_matrix(args.workload, rank, barrier)
    n_genes, n = coo.shape
    perms_total = args.perms or synth.CONFIGS[args.workload][4]
    if args.scaling == "strong":
        from pangenomix_b200.distributed import shard_bounds
        lo, hi = shard_bounds(perms_total, world, rank)            # contiguous blocks, as the multi-GPU API shards
        perms_n = hi - lo
        perms_all = perms_total
    else:
        perms_n = perms_total
        perms_all = perms_total * world
    t = time.time()
    eng = engine.PanCoreEngine(coo, device=device)
    hp = eng.host_plan
    log("[bench r%d] plan: %d list rows (%d tasks, %d folded indices), %d bitmap rows, %d perms per list CTA, %.1fs" % (
        rank, hp.n_rows, hp.n_tasks, hp.folded_nnz, hp.n_long, hp.perms_per_cta, time.time() - t))

    # every rank rarefies its own permutations (numpy legacy stream, seed 12345 + rank)
    h_perms, h_perms_owner = engine.pinned_empty((perms_n, n), np.uint16)
    t = time.time()
    if args.scaling == "strong":
        np.random.seed(12345)                     # ONE stream, sharded in contiguous blocks like the multi-GPU API
        h_perms[:] = engine.draw_legacy_permutations(n, perms_total)[lo:hi]
    else:
        np.random.seed(12345 + rank)
        engine.draw_legacy_permutations(n, perms_n, out=h_perms)
    host_rng_s = time.time() - t
    d_perms = torch.empty((perms_n, n), dtype=torch.int16, device=device)
    d_perms.copy_(h_perms_owner)
    # N > 1: the curves of step i travel to rank 0 (NCCL gather over NVLink, asynchronous) while
    # step i + 1 is computed into the other buffer; the timed region ends when every gather has landed.
    n_buf = 2 if world > 1 else 1
    d_outs = [torch.empty((perms_n, 2 * n), dtype=torch.int32, device=device) for _ in range(n_buf)]
    d_out = d_outs[0]
    gather = None
    if world > 1:
        from pangenomix_b200.distributed import CurveGather, shard_bounds as _sb
        rows_max = _sb(perms_total, world, 0)[1] if args.scaling == "strong" else perms_n
        if rows_max != perms_n:                  # ragged strong-scaling shards: the gather moves equal blocks
            d_outs = [torch.zeros((rows_max, 2 * n), dtype=torch.int32, device=device) for _ in range(n_buf)]
        gather = CurveGather(rows_max, 2 * n, device, dst=0, n_buffers=n_buf,
                             prefer_peer=os.environ.get("PGX_GATHER", "peer") != "nccl")
        log("[bench r%d] curve gather: %s%s" % (rank, gather.mode,
                                                 "" if gather.mode == "peer-push" else " (%s)" % getattr(gather, "fallback_reason", "requested")))
    step_no = [0]

    def step():
        b = step_no[0] % n_buf
        step_no[0] += 1
        if gather is not None:
            gather.before_overwrite(b)        # the buffer's previous transfer has read it
        eng.curves_device(d_perms, out=d_outs[b][:perms_n])
        if gather is not None:
            gather.send(b, d_outs[b])

    def drain():
        if gather is not None:
            gather.drain()

    for _ in range(max(args.warmup, 3)):
        step()
    drain()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    time.sleep(0.2)
    launches0 = _native.launch_count()
    barrier()
    torch.cuda.synchronize()
    # Timing hygiene: the inputs of a step must not be served from L2 by the previous step.  Big workloads
    # (C4, C5) stream more than L2 per step by themselves; small ones (C1, C2) get an L2 flush -- a
    # 256 MB memset -- between steps, outside the per-step CUDA-event brackets.
    step_bytes = d_perms.numel() * 2 + d_out.numel() * 4
    flush = None
    if step_bytes < 2 * l2_bytes:
        flush = torch.empty(max(256 << 20, 2 * l2_bytes), dtype=torch.uint8, device=device)
    w0 = time.perf_counter()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        drain()
        e1.record()
        torch.cuda.synchronize()
        elapsed = e0.elapsed_time(e1)
    else:
        brackets = []
        for _ in range(args.steps):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step()
            drain()
            b.record()
            brackets.append((a, b))
        torch.cuda.synchronize()
        elapsed = sum(a.elapsed_time(b) for a, b in brackets)
    w1 = time.perf_counter()
    if args.dump_outputs and rank == 0:
        # the curves of the last timed step, before the profile pass below overwrites the buffer
        last = d_outs[(step_no[0] - 1) % n_buf][:perms_n]
        rows = dump_rows(perms_n, 2 * n * 8, 2 * n * 8 + 4096)
        sample = last.index_select(0, torch.from_numpy(rows).to(device)).double().cpu().numpy()
        mean = (last.sum(dim=0, dtype=torch.int64).double() / perms_n).cpu().numpy()
        dump_outputs(args.dump_outputs, {"curves": sample, "curve_rows": rows.astype(np.float64), "mean_curve": mean})
    barrier()
    ms = torch.tensor([elapsed], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    launches = _native.launch_count() - launches0
    clocks = sampler.window(w0, w1) if sampler else None

    # per-kernel durations for the roofline: a separate pass with CUDA events around every kernel
    # (the library then runs the two row kernels back to back instead of side by side)
    _native.profile_read()
    _native.profile_enable(True)
    d_out = d_outs[0][:perms_n]
    for _ in range(min(args.steps, 3)):
        eng.curves_device(d_perms, out=d_out)
    torch.cuda.synchronize()
    list_ms, probe_ms, scan_ms, calls = _native.profile_read()
    row_ms = list_ms + probe_ms
    _native.profile_enable(False)
    ms_per_step = ms_total / args.steps

    # the gathered blocks really are on rank 0 (its own block bit for bit, the others by invariants)
    if gather is not None:
        barrier()
        if rank == 0:
            b_last = (step_no[0] - 1) % n_buf
            got = gather.gathered(b_last)
            assert torch.equal(got[0], d_outs[b_last])
            far = got[world - 1][:min(16, perms_n)].cpu().numpy()
            assert np.all(np.diff(far[:, :n], axis=1) >= 0) and np.array_equal(far[:, 0], far[:, n])
            assert far[:, n - 1].min() > 0 and not np.array_equal(far, d_outs[b_last][:min(16, perms_n)].cpu().numpy())
        barrier()

    # parity guard on the timed output (size-independent invariants, cheap)
    curves = d_out[:64].cpu().numpy()
    h_check = curves
    assert np.all(np.diff(curves[:, :n], axis=1) >= 0) and np.all(np.diff(curves[:, n:], axis=1) <= 0)
    assert np.array_equal(curves[:, 0], curves[:, n])

    # ---- end to end through the host-buffer C-ABI call ----
    e2e = None
    if not args.no_e2e:
        h_out, h_out_owner = engine.pinned_empty((perms_n, 2 * n), np.int32)
        for _ in range(2):
            eng.curves_host(h_perms, out=h_out)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            eng.curves_host(h_perms, out=h_out)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
        barrier()
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        assert np.array_equal(h_out[:64], curves)
        packed = 0 < eng.c_plan.max_colsum <= 65535 and not os.environ.get("PGX_WIDE_BINS")
        head = int(_native.load().pgx_split_head()) if packed else 0
        row_bytes = (2 * n + 2 * head) if head > 0 else (4 * n if packed else 8 * n)
        e2e = {"value": perms_all * args.steps / float(dt.item()), "unit": UNIT,
               "h2d_bytes_per_step": 2 * n * perms_all, "d2h_bytes_per_step": row_bytes * perms_all,
               "ms_per_step": float(dt.item()) / args.steps * 1e3,
               "path": "pgx_pan_core_curves_host: pinned uint16 permutations in, int32 curves out in host memory, wall clock; "
                       + (("the device ships the curves' steps, the first %d of each curve as uint16 and the rest as uint8 "
                           "(%d bytes per permutation), host threads rebuild the int32 curves in the caller's buffer inside "
                           "the timed region" % (head, row_bytes)) if head > 0 else
                          "the device ships the curves' uint16 steps (4N bytes per permutation), host threads rebuild the "
                          "int32 curves in the caller's buffer inside the timed region" if packed else
                          "int32 curves cross PCIe as they are (a genome holds more than 65,535 genes)"),
               "host_rng_s_per_step_not_included": host_rng_s}
        del h_out, h_out_owner
    if sampler:
        sampler.stop()

    # ---- the reference-facing Python call itself: RNG draws + upload + kernels + float64 DataFrame ----
    api = None
    if rank == 0 and not args.no_e2e:
        import contextlib
        import io
        from pangenomix_b200 import pangenome_analysis as pa, sparse_utils as su
        index, columns = synth.labels_for(n_genes, n)
        lsdf = su.LightSparseDataFrame(index, columns, coo)
        pa._ENGINE_CACHE[lsdf] = (lsdf.data, eng, pa._fingerprint(lsdf.data))              # "uploaded once": reuse the resident table
        iters = int(min(perms_n, 2000))
        np.random.seed(12345)
        with contextlib.redirect_stdout(io.StringIO()):
            pa.estimate_pan_core_size(lsdf, min(iters, 64))
            np.random.seed(12345)
            t0 = time.perf_counter()
            df = pa.estimate_pan_core_size(lsdf, iters)
            api_s = time.perf_counter() - t0
        np.random.seed(12345)
        t0 = time.perf_counter()
        engine.draw_legacy_permutations(n, iters)
        rng_s = time.perf_counter() - t0
        # the first call on a table a user has on disk: read_lsdf (inflate + labels) + plan + upload + curves
        import tempfile
        npz = os.path.join(tempfile.gettempdir(), "pgx_bench_%s.npz" % args.workload)
        if not os.path.exists(npz):
            lsdf.to_npz(npz)
        t0 = time.perf_counter()
        cold = su.read_lsdf(npz)
        t_read = time.perf_counter() - t0
        np.random.seed(12345)
        with contextlib.redirect_stdout(io.StringIO()):
            df_cold = pa.estimate_pan_core_size(cold, 64)
        t_cold = time.perf_counter() - t0
        assert np.array_equal(df_cold.values, df.values[:64])
        api_cold = {"call": "read_lsdf(npz) + estimate_pan_core_size(df_genes, 64) on a table not seen before",
                    "seconds": t_cold, "read_lsdf_seconds": t_read, "plan_upload_first_call_seconds": t_cold - t_read,
                    "npz_bytes": os.path.getsize(npz)}
        del cold, df_cold
        assert df.shape == (iters, 2 * n) and df.values.dtype == np.float64
        assert np.array_equal(df.values[:8].astype(np.int32), h_check[:8]) if iters >= 8 else True
        api = {"call": "pangenomix_b200.pangenome_analysis.estimate_pan_core_size(df_genes, %d)" % iters,
               "value": iters / api_s, "unit": UNIT, "seconds": api_s,
               "host_rng_seconds": rng_s, "host_rng_perms_per_s": iters / rng_s,
               "note": "includes the %d numpy-legacy shuffles drawn on the host (bit-exact RNG stream), "
                       "H2D/D2H and the float64 DataFrame; the table was already resident" % iters,
               "cold": api_cold}
        del df

    # ---- next row of the scope table: Heaps-law fits of every curve of the step, on the device ----
    heaps = None
    if rank == 0 and not args.no_e2e:
        import warnings
        import pandas as pd
        from pangenomix_b200 import pangenome_analysis as pa
        engine.fit_heaps_device(d_out[:8])
        torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        fit, info = engine.fit_heaps_device(d_out)
        h1.record()
        torch.cuda.synchronize()
        fit_ms = h0.elapsed_time(h1)
        sample = d_out[:3].cpu().numpy().astype(np.float64)
        cols = ["Pan%d" % (i + 1) for i in range(n)] + ["Core%d" % (i + 1) for i in range(n)]
        t0 = time.perf_counter()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want = pa.fit_heaps_by_iteration(pd.DataFrame(sample, columns=cols))
        scipy_s = (time.perf_counter() - t0) / 3
        np.testing.assert_allclose(fit[:3].cpu().numpy(), want.values, rtol=5e-6)
        heaps = {"call": "pgx_heaps_fit on the %d device-resident curves of one step (%d points each)" % (perms_n, n),
                 "value": perms_n / (fit_ms / 1e3), "unit": "fits/s", "ms": fit_ms,
                 "converged": int((info > 0).sum().item()),
                 "scipy_curve_fit_fits_per_s": 1.0 / scipy_s,
                 "note": "fit_heaps_by_iteration (scipy curve_fit, one host core) timed on 3 of the same curves; "
                         "results agree to 5e-6 relative (scipy's stopping tolerance)"}

    # ---- last row of the scope table (8f rank 4): gene-frequency spectrum + beta-binomial core estimate ----
    beta_binomial = None
    if rank == 0 and not args.no_e2e:
        beta_binomial = beta_binomial_entry(coo, check=not args.no_cpu_baseline)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = perms_all * args.steps / (ms_total / 1e3)
    peak, peak_src = measured_peak()
    a_perm = hp.algorithmic_bytes_per_perm
    calls = max(1, calls)
    # dominant kernel: the slower of the two row kernels
    kind = "list" if list_ms >= probe_ms else "probe"
    k_ms = (list_ms if kind == "list" else probe_ms) / calls
    k_bytes = hp.algorithmic_bytes_of(kind)
    hbm_achieved = k_bytes * perms_n / (k_ms / 1e3) / 1e9 if k_ms > 0 else None
    combined = a_perm * perms_n / (row_ms / calls / 1e3) / 1e9 if row_ms > 0 else None
    ncu = ncu_counters(args.workload, kind)
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    sm_count = int(_native.device_info()["sm_count"])
    kernel_name = "list_kernel<%d>" % hp.perms_per_cta if kind == "list" else "probe_kernel<%d>" % hp.slice_words
    if kind == "list":
        # What binds the list kernel is the shared-memory / LSU data pipe of the SMs (one 128-byte wavefront per
        # clock per SM), not HBM: every folded index is ONE shared-memory gather of 2 bytes per permutation.
        smem_peak = 128.0 * sm_count * sm_mhz * 1e6 / 1e9
        wf = ncu.get("lsu_wavefronts_per_perm")
        achieved = wf * 128.0 * perms_n / (k_ms / 1e3) / 1e9 if wf and k_ms > 0 else None
        roofline = {
            "bound": "smem_lsu", "kernel": kernel_name, "achieved": achieved, "peak": smem_peak, "unit": "GB/s",
            "frac": achieved / smem_peak if achieved else None,
            "traffic": wf * 128.0 * perms_n if wf else None,
            "peak_source": "128 B per clock per SM x %d SMs x %.0f MHz (SM clock sampled during the timed region)" % (sm_count, sm_mhz),
            "pipe_utilisation_under_ncu": (ncu.get("lsu_pipe_pct_of_peak") or 0) / 100.0 or None,
            "wavefronts_per_lds128": ncu.get("wavefronts_per_shared_load"),
            "algorithmic_smem_bytes_per_perm": 2 * hp.folded_nnz,
            "algorithmic_frac": 2.0 * hp.folded_nnz * perms_n / (k_ms / 1e3) / 1e9 / smem_peak if k_ms > 0 else None,
            "note": "achieved = LSU data-pipe wavefronts of the kernel (ncu capture at HEAD, %s) x 128 B / live CUDA-event "
                    "duration; the wavefronts are shared-memory gathers (one LDS.128 per folded index per %d permutations), "
                    "histogram REDs, chunk loads and rank-table stores; algorithmic_frac counts only 2 bytes per (folded index, "
                    "permutation)" % (ncu.get("source", "none committed"), hp.perms_per_cta),
        }
    else:
        issue = (ncu.get("issue_active_pct") or 0) / 100.0 or None
        roofline = {
            "bound": "issue", "kernel": kernel_name, "achieved": issue, "peak": 1.0, "unit": "fraction of issue slots",
            "frac": issue, "traffic": None, "peak_source": "ncu smsp__issue_active (%s)" % ncu.get("source", "none committed"),
            "alu_pipe_utilisation_under_ncu": (ncu.get("alu_pipe_pct") or 0) / 100.0 or None,
        }
    dram = ncu.get("dram_bytes_per_perm")
    roofline.update({
        "perms_per_launch": perms_n, "ms_per_launch": k_ms,
        "list_ms_per_launch": list_ms / calls, "probe_ms_per_launch": probe_ms / calls,
        "prep_and_scan_ms_per_launch": scan_ms / calls,
        "row_kernels_serialised_ms_per_launch": row_ms / calls,
        "step_ms_with_kernels_overlapped": ms_per_step,
        "list_rows": hp.n_rows, "bitmap_rows": hp.n_long, "long_threshold": hp.long_threshold,
        # SURVEY.md section 8d's bookkeeping, kept beside the physical bound: one pass over the canonical int32
        # gene-major CSR per permutation.  The kernels never move those bytes (2-byte folded indices once per %d
        # permutations, bitmaps shared by 1,024 W genes), so this fraction is an EFFECTIVE one and exceeds 1.
        "hbm": {"peak": peak, "peak_source": peak_src, "unit": "GB/s",
                "algorithmic_bytes_per_perm": k_bytes, "algorithmic_bytes_per_perm_whole_table": a_perm,
                "achieved_algorithmic": hbm_achieved, "effective_frac": hbm_achieved / peak if hbm_achieved else None,
                "row_kernels_effective_frac_whole_table": combined / peak if combined else None,
                "traffic": dram * perms_n if dram else None,
                "dram_frac": dram * perms_n / (k_ms / 1e3) / 1e9 / peak if dram and k_ms > 0 else None,
                "streamed_bytes_per_row_pass": hp.streamed_bytes_per_pass},
    })
    cpu = None
    if (world == 1 or args.cpu_check) and not args.no_cpu_baseline:
        from oracle import cport
        threads = os.cpu_count() or 1
        gm, sample_perms, t1 = cpu_sample(coo, n, args.cpu_seconds, threads)
        t0 = time.perf_counter()
        pan, core = cport.curves_direct(gm, sample_perms, n_threads=threads)
        dt = time.perf_counter() - t0
        # the CPU arm doubles as a checker of the GPU result on its sample
        check = eng.curves_host(sample_perms[:threads].astype(np.uint16))
        assert np.array_equal(check, np.hstack([pan, core])[:threads].astype(np.int32)), "GPU != oracle"
        cpu = {"value": sample_perms.shape[0] / dt, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "%d permutations of the same table (of %d), oracle C port of "
                         "pangenome_analysis.py:81-90, %d threads" % (sample_perms.shape[0], perms_n, threads),
               "single_thread_s_per_perm": t1,
               "reference_python": python_reference_sample(coo, eng, n_iter=1 if n >= 2000 else 20)
               if coo.shape[0] * coo.shape[1] <= 4e9 else {"skipped": "one permutation of this table takes the Python reference about 10 minutes"}}
    config = workload_config(args.workload, coo, perms_total, world, args.scaling)
    if flush is None:
        config["l2_policy"] = "inputs larger than L2: %.0f MB of permutations + %.0f MB of curves + %.0f MB of folded rows per step" % (
            d_perms.numel() * 2 / 1e6, d_out.numel() * 4 / 1e6, hp.streamed_bytes_per_pass / 1e6)
    else:
        config["l2_policy"] = ("L2 flushed (%.0f MB memset) between timed steps, every step timed with its own CUDA events: "
                               "%.1f MB of permutations + %.1f MB of curves + %.1f MB of folded rows per step fit L2" % (
                                   flush.numel() / 1e6, d_perms.numel() * 2 / 1e6, d_out.numel() * 4 / 1e6,
                                   hp.streamed_bytes_per_pass / 1e6))
    if world > 1 and gather.mode == "peer-push":
        config["gather"] = ("int32 curves of every rank pushed into rank 0's symmetric-memory buffer over NVLink "
                            "(copy-engine peer copies on a side stream) inside the timed region, overlapped with "
                            "the next step (two buffers)")
    elif world > 1:
        config["gather"] = ("NCCL gather of int32 curves to rank 0 inside the timed region, asynchronous, "
                            "overlapped with the next step (two output buffers)")
    else:
        config["gather"] = "none (1 GPU)"
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "u16", "data": "synthetic", "config": config,
        "cells_per_s": value * n_genes * n, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": int(launches), "clocks": clocks, "host_rng_s_for_perms": host_rng_s, "api": api, "heaps": heaps,
        "beta_binomial": beta_binomial,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def beta_binomial_entry(coo, check=True, num_points=100, ks_iter=1000):
    """compute_beta_binomial_core_genome on the workload's table (SURVEY.md 8f rank 4): the table's marginals and
    gene-frequency spectrum counted on the GPU, then the fit with the reference's default 1,000 Monte-Carlo KS
    iterations on the GPU.  With ``check`` the reference's own simulation loop (pangenome_analysis.py:471-480,
    restated in oracle/betabin_np.py) is timed on a few iterations of the same stream and compared bit for bit."""
    import warnings
    import pandas as pd
    from pangenomix_b200 import engine
    from pangenomix_b200 import pangenome_analysis as pa
    n_genes, n = coo.shape
    try:
        engine.table_marginals(coo)                                   # staging, first-call costs
        t0 = time.perf_counter()
        row_sum, col_sum, spectrum, _ = engine.table_marginals(coo)
        marg_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        want_row = np.asarray(coo.sum(axis=1)).ravel()
        want_col = np.asarray(coo.sum(axis=0)).ravel()
        scipy_s = time.perf_counter() - t0
        assert np.array_equal(row_sum, want_row) and np.array_equal(col_sum, want_col)
        freqs = np.flatnonzero(spectrum[1:]) + 1
        counts = pd.Series(spectrum[freqs], index=freqs)                  # ascending gene frequency
        calls = []
        original = engine.ks_montecarlo_statistics

        def timed(choice_cdf, model_cdf, n_samples, iterations, device=None):
            state = np.random.get_state()
            t = time.perf_counter()
            out = original(choice_cdf, model_cdf, n_samples, iterations, device=device)
            calls.append({"seconds": time.perf_counter() - t, "n_samples": int(n_samples), "iterations": int(iterations),
                          "sim_limit": int(len(model_cdf)), "state": state, "cdf": choice_cdf, "model": model_cdf,
                          "ks_sim": out})
            return out

        engine.ks_montecarlo_statistics = timed
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                np.random.seed(12345)
                pa.compute_beta_binomial_core_genome(None, df_counts=counts, num_points=num_points, ks_iter=8)   # staging
                del calls[:]
                np.random.seed(12345)
                t0 = time.perf_counter()
                fit = pa.compute_beta_binomial_core_genome(None, df_counts=counts, num_points=num_points, ks_iter=ks_iter)
                fit_s = time.perf_counter() - t0
        finally:
            engine.ks_montecarlo_statistics = original
        entry = {"call": "table_marginals + compute_beta_binomial_core_genome(df_counts=spectrum, num_points=%d, ks_iter=%d)"
                         % (num_points, ks_iter),
                 "marginals_ms": marg_s * 1e3, "scipy_sum_both_axes_ms": scipy_s * 1e3,
                 "fit_seconds": fit_s, "fit": {k: (None if v != v else float(v)) for k, v in fit.items()}}
        if calls:
            c = calls[0]
            draws = c["n_samples"] * c["iterations"]
            entry.update({"ks_seconds": c["seconds"], "ks_draws": draws, "ks_draws_per_s": draws / c["seconds"],
                          "ks_n_samples": c["n_samples"], "ks_sim_limit": c["sim_limit"]})
            if check:
                from oracle import betabin_np as ob
                it_ref = max(2, min(c["iterations"], int(3e6 // max(1, c["n_samples"]))))
                raw, _ = ob.raw_words(c["state"], 2 * c["n_samples"] * it_ref)
                t0 = time.perf_counter()
                draws_ref = np.asarray(c["cdf"]).searchsorted(ob.uniforms_from_raw(raw), side="right").reshape(it_ref, c["n_samples"])
                ks_ref = np.zeros(it_ref)
                for i in np.arange(it_ref):                                # the loop of :475-479, as written there
                    vals, cnts = np.unique(draws_ref[i, :], return_counts=True)
                    pmf = np.zeros(c["sim_limit"])
                    for j in np.arange(len(vals)):
                        pmf[vals[j]] += cnts[j]
                    ks_ref[i] = np.max(np.abs(np.cumsum(pmf) / pmf.sum() - c["model"]))
                ref_s = time.perf_counter() - t0
                assert np.array_equal(c["ks_sim"][:it_ref], ks_ref)
                entry["reference_loop"] = {"draws_per_s": c["n_samples"] * it_ref / ref_s, "iterations": it_ref, "kind": "port",
                                           "note": "searchsorted + np.unique + eCDF loop per iteration on one host core, raw stream "
                                                   "already drawn; first %d statistics identical to the GPU's" % it_ref}
        # throughput of the simulation at a size that fills the device: as many draws per iteration as the table has
        # genes (every gene a core gene), the reference's default 1,000 iterations
        from scipy.special import betaln
        sim_limit, big_n = 128, int(min(n_genes, 200_000))
        k = np.arange(sim_limit, dtype=np.float64)
        pmf = np.exp(-np.log(n + 1) - betaln(n - k + 1, k + 1) + betaln(k + 0.5, n - k + 60.0 * n / 300.0) - betaln(0.5, 60.0 * n / 300.0))
        model_cdf = np.cumsum(pmf)
        cdf = (pmf / pmf.sum()).cumsum()
        cdf /= cdf[-1]
        np.random.seed(1)
        engine.ks_montecarlo_statistics(cdf, model_cdf, big_n, 8)
        t0 = time.perf_counter()
        engine.ks_montecarlo_statistics(cdf, model_cdf, big_n, ks_iter)
        big_s = time.perf_counter() - t0
        entry.update({"value": big_n * ks_iter / big_s, "unit": "draws/s",
                      "value_is": "ks_montecarlo_statistics: %d iterations of %d draws over %d bins through the host-buffer call "
                                  "(bit-exact MT19937 stream drawn on the host inside the timed region)" % (ks_iter, big_n, sim_limit)})
        return entry
    except Exception as exc:                                         # noqa: BLE001 - an auxiliary entry never fails the bench
        return {"error": "%s: %s" % (type(exc).__name__, exc)}


# --------------------------------------------------------------------------------------
# Bernoulli grid (config C3): LL + gradient evaluations per second
# --------------------------------------------------------------------------------------
def bernoulli_roofline(g, n, absent, evals_per_s, alg_bytes, hbm_peak, hbm_src):
    """The Bernoulli grid kernel is bound by the fp64 pipe (one log and one reciprocal per ABSENT cell on an
    L2-resident 1-bit table), not by HBM: frac is the fp64 pipe utilisation of the committed ncu capture; the HBM
    bookkeeping (table + P, Q, gradient once per evaluation) is kept as an effective fraction."""
    ncu = ncu_counters("c3", "grid")
    frac = (ncu.get("fp64_pipe_pct") or 0) / 100.0 or None
    return {"bound": "fp64_pipe", "kernel": "bernoulli grid_kernel", "achieved": frac, "peak": 1.0,
            "unit": "fraction of fp64 pipe cycles", "frac": frac, "traffic": ncu.get("dram_bytes_per_perm"),
            "peak_source": "ncu sm__inst_executed_pipe_fp64 (%s)" % ncu.get("source", "none committed"),
            "issue_active_under_ncu": (ncu.get("issue_active_pct") or 0) / 100.0 or None,
            "active_lanes_per_instruction": ncu.get("active_lanes_per_instruction"),
            "absent_cells_per_s": evals_per_s * absent,
            "hbm": {"peak": hbm_peak, "peak_source": hbm_src, "unit": "GB/s", "algorithmic_bytes_per_eval": alg_bytes,
                    "achieved_algorithmic": alg_bytes * evals_per_s / 1e9, "effective_frac": alg_bytes * evals_per_s / 1e9 / hbm_peak}}


def run_bernoulli(args):
    """C3 of BASELINE.json: compute_bernoulli_grid_core_genome on 400 genomes.  A step is one
    evaluation of the log-likelihood AND its gradient at a new (P, Q) -- what one L-BFGS-B iteration
    of pangenome_analysis.py:156-160 costs.  value: table, P, Q resident on the device; e2e: through
    BernoulliGrid.ll_grad (host P,Q in, host LL + gradient out); cpu_baseline: the reference's own
    numpy expressions (:244-266, restated in oracle/pancore_np.py) on the same table."""
    import ctypes
    import torch
    import oracle
    from pangenomix_b200 import _native, engine, synth
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(0)
    g, n = args.genes, 400
    x, _, _ = synth.bernoulli_grid_matrix(g, n, seed=3)
    grid = engine.BernoulliGrid(x, device="cuda:0")
    rng = np.random.RandomState(1)
    lo, hi = 0.8, 0.99999999
    n_pts = 8
    pts = [np.concatenate((rng.uniform(lo, hi, g), rng.uniform(lo, hi, n))) for _ in range(n_pts)]
    d_pts = [torch.from_numpy(p).cuda() for p in pts]
    lib = _native.load()
    stream = torch.cuda.current_stream().cuda_stream

    def launch(d_pq):
        _native.check(lib.pgx_bernoulli_ll_grad(
            grid._xbits.data_ptr(), grid.words_per_row, g, n, grid._row_count.data_ptr(),
            grid._col_count.data_ptr(), d_pq.data_ptr(), d_pq.data_ptr() + 8 * g,
            grid._res.data_ptr(), grid._res.data_ptr() + 8, grid._scratch.data_ptr(), stream))

    for i in range(max(args.warmup, 3)):
        launch(d_pts[i % n_pts])
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    time.sleep(0.2)
    steps = args.steps
    launches0 = _native.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    for i in range(steps):
        launch(d_pts[i % n_pts])
    e1.record()
    torch.cuda.synchronize()
    w1 = time.perf_counter()
    if args.dump_outputs:
        res = grid._res.cpu().numpy()                 # [LL, gradient] at the point of the last step
        dump_outputs(args.dump_outputs, {"loglikelihood": res[:1], "gradient": res[1:]})
    ms = e0.elapsed_time(e1)
    launches = _native.launch_count() - launches0
    clocks = sampler.window(w0, w1)
    # end to end through the Python engine (pinned staging, H2D of P,Q, D2H of LL + gradient)
    for i in range(3):
        grid.ll_grad(pts[i])
    t0 = time.perf_counter()
    for i in range(steps):
        ll, grad = grid.ll_grad(pts[i % n_pts] + (i // n_pts) * 1e-12)     # defeat the value cache
    e2e_s = time.perf_counter() - t0
    sampler.stop()
    # CPU: the reference's numpy expressions, and parity on this very point
    t0 = time.perf_counter()
    ref_ll = oracle.bernoulli_ll(x, pts[0][:g], pts[0][g:])
    ref_grad = oracle.bernoulli_grad(x, pts[0][:g], pts[0][g:])
    cpu_s = time.perf_counter() - t0
    got_ll, got_grad = grid.ll_grad(pts[0])
    np.testing.assert_allclose(got_ll, ref_ll, rtol=1e-9)
    np.testing.assert_allclose(got_grad, ref_grad, rtol=1e-9, atol=1e-9 * np.abs(ref_grad).max())
    # the reference-facing call itself: the whole L-BFGS-B fit (scipy on the host drives the kernels),
    # and the same fit with the reference's numpy likelihood on one core (bounded: 4,000 genes)
    import contextlib
    import io
    import warnings
    import pandas as pd
    import scipy.optimize
    from pangenomix_b200 import pangenome_analysis as pa
    index, columns = synth.labels_for(g, n)
    df_dense = pd.DataFrame(x, index=index, columns=columns)
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        df_opt, res = pa.compute_bernoulli_grid_core_genome(df_dense)
        fit_s = time.perf_counter() - t0
    fit = {"call": "compute_bernoulli_grid_core_genome(df %d x %d)" % (g, n), "seconds": fit_s,
           "iterations": int(res.nit), "evaluations": int(res.nfev), "final_loglikelihood": float(-res.fun),
           "message": str(res.message)}
    g_ref = min(g, 4000)
    x_ref = x[:g_ref]
    p0 = np.clip(np.concatenate((x_ref.sum(axis=1) / float(n), 0.9999 * np.ones(n))), 0.8, 0.99999999)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        ref = scipy.optimize.minimize(lambda v: -oracle.bernoulli_ll(x_ref, v[:g_ref], v[g_ref:]), p0, method="L-BFGS-B",
                                      jac=lambda v: -oracle.bernoulli_grad(x_ref, v[:g_ref], v[g_ref:]),
                                      bounds=[(0.8, 0.99999999)] * (g_ref + n))
        ref_s = time.perf_counter() - t0
    fit["reference_numpy_fit_seconds_%d_genes" % g_ref] = ref_s
    fit["reference_numpy_fit_iterations"] = int(ref.nit)
    if g_ref == g:
        fit["optimum_rel_diff_vs_reference"] = float(abs(res.fun - ref.fun) / abs(ref.fun))

    absent = int(x.size - x.sum())
    value = steps / (ms / 1e3)
    peak, peak_src = measured_peak()
    alg_bytes = g * ((n + 31) // 32) * 4 + 8 * (g + n) * 2 + 8
    line = {
        "metric": "bernoulli_grid_ll_grad_evals_per_sec", "value": value, "unit": "evals/s", "n_gpus": 1,
        "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C3: compute_bernoulli_grid_core_genome likelihood + gradient on a synthetic %d-gene x "
                               "400-genome dense 0/1 table (prob_bounds 0.8..0.99999999), one evaluation per step" % g,
                   "n_genes": g, "n_genomes": n, "absent_cells": absent,
                   "l2_policy": "%d distinct (P, Q) points cycled; the 1-bit table (%.1f MB) is L2-resident by design" % (
                       n_pts, g * ((n + 31) // 32) * 4 / 1e6)},
        "cells_per_s": value * g * n, "absent_cells_per_s": value * absent,
        "roofline": bernoulli_roofline(g, n, absent, value, alg_bytes, peak, peak_src),
        "cpu_baseline": {"value": 1.0 / cpu_s, "unit": "evals/s", "cores": 1, "kind": "port",
                         "sample": "one LL + gradient evaluation of the same table with the reference's numpy "
                                   "expressions (pangenome_analysis.py:244-266), single-threaded as in the reference"},
        "e2e": {"value": steps / e2e_s, "unit": "evals/s", "h2d_bytes_per_step": 8 * (g + n),
                "d2h_bytes_per_step": 8 * (g + n + 1), "ms_per_step": e2e_s / steps * 1e3,
                "path": "BernoulliGrid.ll_grad: pinned P,Q up, 2 kernels, LL + gradient down"},
        "gpu_launches": int(launches), "clocks": clocks,
        "fit": fit,
        "parity": {"ll_rel_err": abs(got_ll - ref_ll) / abs(ref_ll),
                   "grad_max_rel_err": float(np.max(np.abs(got_grad - ref_grad)) / np.abs(ref_grad).max())},
    }
    emit(line)


_JSON_OUT = None


def emit(line):
    """The one JSON line goes to the real stdout; everything else any library prints (NCCL's
    version banner, ...) was redirected to stderr in main()."""
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def main():
    global _JSON_OUT
    args = parse_args()
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)                                  # fd 1 -> stderr for C libraries and stray prints
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if world != args.gpus:
        log("[bench] note: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE" % (args.gpus, world))
    if args.workload == "c3":
        if rank == 0:
            run_bernoulli(args)
    elif args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
