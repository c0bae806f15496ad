"""Shared-gene matrix (pgx_shared_genes) and genomic fluidity on one GPU, phase by phase, with a scipy CPU arm.

    python scripts/probe_shared_genes.py [--configs c4,c5] [--steps 10] [--warmup 2] [--out DIR]

Per config, on a cached engine (the table planned and uploaded once):
  phases     device time of every kernel of one pgx_shared_genes + pgx_fluidity_rows call, from torch.profiler with
             CUDA activities in a pass of its own, averaged over ``steps`` calls: init (count kernels + closed forms),
             scatter (list-row pairs), expand (bitmap rows -> E), gemm (tcgen05 S += E E^T), mirror, rows
  gemm rate  8-bit integer operations of the tiles the GEMM computes (2 x 128 x 256 x K per tile) over its time,
             against 4.5 POPS (NVIDIA's dense INT8 figure for one B200: a sixteenth of the 72 POPS it prints for
             eight GPUs with sparsity); the upper triangle's own share of those operations is printed beside it
  call       CUDA events around shared_genes_device + fluidity_rows_device (workspace allocation included)
  api        compute_genomic_fluidity end to end (host clock; its result comes back to the host)
  cpu        scipy X[:, c]^T X for a sample of genomes c on the host, extrapolated to all N rows (labelled so), and
             the whole product where --cpu-full-max-genomes allows it
The card's name, power limit and maximum SM clock are read in the same run.  Writes DIR/shared_genes_<configs>.json
and DIR/shared_genes_<configs>.log (default DIR: profiles/r04).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "scripts"))

from probe_pan_core_summary import card, load  # noqa: E402

INT8_DENSE_OPS = 4.5e15
PHASES = (("init", ("shared_count", "shared_full", "shared_init")), ("scatter", ("shared_pairs",)),
          ("expand", ("shared_expand",)), ("gemm", ("shared_gemm",)), ("mirror", ("shared_mirror",)),
          ("rows", ("fluidity_rows",)))


def gemm_counts(hp):
    """(ops of the computed tiles, ops of the strict upper triangle) of the GEMM: 2 per multiply-add."""
    n = hp.n_genomes
    k = hp.n_superblocks * 1024 * hp.slice_words if hp.n_long else 0
    row_tiles, col_tiles = (n + 127) // 128, (n + 255) // 256
    tiles = sum(col_tiles - rb // 2 for rb in range(row_tiles))
    return 2.0 * tiles * 128 * 256 * k, 2.0 * (n * (n - 1) / 2) * hp.n_long


def phase_times(torch, eng, steps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            eng.fluidity_rows_device(eng.shared_genes_device())
        torch.cuda.synchronize()
    out = {name: 0.0 for name, _ in PHASES}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        us = ev.cuda_time_total if us is None else us
        for name, keys in PHASES:
            if any(k in ev.key for k in keys):
                out[name] += us / 1000.0 / steps
    return out


def run_config(name, args, log):
    import torch
    from pangenomix_b200 import engine, pangenome_analysis as pa, sparse_utils as su, synth
    from oracle import shared_np
    coo = load(name)
    n_genes, n = coo.shape
    df = su.LightSparseDataFrame(*synth.labels_for(n_genes, n), coo)
    eng = pa._engine_for(df)
    hp = eng.host_plan
    res = {"config": name, "n_genes": n_genes, "n_genomes": n, "n_long": hp.n_long, "n_rows": hp.n_rows,
           "slice_words": hp.slice_words, "pairs": int((hp.row_len.astype(np.int64) * (hp.row_len - 1) // 2).sum()),
           "workspace_bytes": eng.shared_workspace_bytes()}
    log("%s: N = %d, G = %d, bitmap rows %d (GEMM K %d), list rows %d, list-row pairs %.3g, workspace %.2f GB" % (
        name, n, n_genes, hp.n_long, hp.n_superblocks * 1024 * hp.slice_words if hp.n_long else 0, hp.n_rows,
        res["pairs"], res["workspace_bytes"] / 1e9))

    for _ in range(args.warmup):
        eng.fluidity_rows_device(eng.shared_genes_device())
    torch.cuda.synchronize()
    res["phases_ms"] = phase_times(torch, eng, args.steps)
    log("  phases (ms, profiler device time per call): " + ", ".join("%s %.3f" % kv for kv in res["phases_ms"].items()))
    ops, upper_ops = gemm_counts(hp)
    g = res["phases_ms"]["gemm"]
    if g > 0:
        res["gemm_tops"] = ops / (g * 1e-3) / 1e12
        res["gemm_share_of_4_5_pops"] = ops / (g * 1e-3) / INT8_DENSE_OPS
        res["gemm_upper_triangle_ops_share"] = upper_ops / ops
        log("  gemm: %.3g ops over the computed tiles in %.3f ms = %.0f TOPS = %.1f %% of 4.5 POPS "
            "(the strict upper triangle is %.1f %% of those ops)" % (
                ops, g, res["gemm_tops"], 100 * res["gemm_share_of_4_5_pops"], 100 * upper_ops / ops))

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        eng.fluidity_rows_device(eng.shared_genes_device())
    e1.record()
    torch.cuda.synchronize()
    res["call_ms"] = e0.elapsed_time(e1) / args.steps
    log("  shared_genes_device + fluidity_rows_device: %.3f ms per call (CUDA events, %d calls)" % (res["call_ms"], args.steps))

    pa.compute_genomic_fluidity(df)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        fl = pa.compute_genomic_fluidity(df)
        times.append((time.perf_counter() - t0) * 1e3)
    res["api_ms_median"], res["api_ms_min"] = float(np.median(times)), float(np.min(times))
    res["fluidity"], res["jackknife_se"] = float(fl["fluidity"]), float(fl["jackknife_se"])
    log("  compute_genomic_fluidity: median %.3f ms, min %.3f ms over %d calls; fluidity %.6f +- %.2e" % (
        res["api_ms_median"], res["api_ms_min"], args.steps, fl["fluidity"], fl["jackknife_se"]))

    # CPU arm: rows of S through scipy for a sample of genomes, checked against the GPU's rows and extrapolated
    cols = np.sort(np.random.default_rng(0).choice(n, min(n, args.cpu_sample), replace=False))
    t0 = time.perf_counter()
    want = shared_np.shared_sample_rows(coo, cols)
    t_sample = time.perf_counter() - t0
    got = eng.shared_genes_device()[torch.from_numpy(cols).to(eng.device)].cpu().numpy()
    res["cpu_sample_rows"] = int(cols.size)
    res["cpu_sample_s"] = t_sample
    res["cpu_extrapolated_s"] = t_sample * n / cols.size
    res["sample_rows_equal"] = bool(np.array_equal(got, want))
    log("  cpu (scipy): %d sampled rows of S in %.2f s -> all %d rows EXTRAPOLATED %.1f s; GPU rows equal: %s" % (
        cols.size, t_sample, n, res["cpu_extrapolated_s"], res["sample_rows_equal"]))
    if n <= args.cpu_full_max_genomes:
        t0 = time.perf_counter()
        shared_np.shared_direct(coo)
        res["cpu_full_s"] = time.perf_counter() - t0
        log("  cpu (scipy): whole X^T X in %.1f s (measured)" % res["cpu_full_s"])
    pa._ENGINE_CACHE.clear()
    del eng
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", default="c4,c5")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cpu-sample", type=int, default=64)
    ap.add_argument("--cpu-full-max-genomes", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r04"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_shared_genes.py needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    tag = args.configs.replace(",", "_")
    lines = []

    def log(msg):
        print(msg, flush=True)
        lines.append(msg)

    info = {"card": card(), "device": torch.cuda.get_device_name()}
    log("card (name, power limit, max SM clock): %s" % info["card"])
    info["results"] = [run_config(name, args, log) for name in args.configs.split(",")]
    with open(os.path.join(args.out, "shared_genes_%s.json" % tag), "w") as f:
        json.dump(info, f, indent=1)
    with open(os.path.join(args.out, "shared_genes_%s.log" % tag), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
