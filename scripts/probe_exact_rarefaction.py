"""Exact pan/core rarefaction (exact_pan_core_summary) on one GPU, phase by phase.

    python scripts/probe_exact_rarefaction.py OUTDIR [--configs c4,c5] [--steps 5] [--warmup 1]

Per config, on a cached engine (the table planned and uploaded once):
  phases     device time of the kernels of one exact_moments_device(std=True) call, from torch.profiler with CUDA
             activities in a pass of its own, averaged over ``steps`` calls: aggregates (vector sums, per-row m / Wp /
             Wa, class counts, closed-form pairs, sort), expand (stored rows -> E panels), gemm (tcgen05 E E^T with the
             histogram epilogue), transform (the moments)
  gemm rate  8-bit integer operations of the launched tiles that compute (2 x 128 x 256 x N_pad per tile) over its
             time, against 4.5 POPS (NVIDIA's dense INT8 figure for one B200)
  api        CUDA events around exact_pan_core_summary with std=False and std=True (result on the host)
  shared     pgx_shared_genes at the same config, phases again, to compare its GEMM rate with the one it had
The card's name, power limit and maximum SM clock are read in the same run.  Writes OUTDIR/exact_<configs>.json and
OUTDIR/exact_<configs>.log.
"""
import argparse
import json
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "scripts"))

from probe_pan_core_summary import card, load  # noqa: E402
from probe_shared_genes import INT8_DENSE_OPS, gemm_counts  # noqa: E402
from probe_shared_genes import phase_times as shared_phase_times  # noqa: E402

PHASES = (("aggregates", ("pair_vectors", "pair_list_rows", "pair_bitmap_rows", "pair_classes", "pair_closed",
                          "pair_scan", "pair_sort", "spectrum_finish")),
          ("expand", ("pair_expand",)), ("gemm", ("pair_hist_gemm",)), ("transform", ("rarefaction_moments",)))


def launched_tiles(rows, panel):
    """(tiles launched, tiles that compute) of every GEMM launch of pgx_pair_overlap_histograms."""
    def triangle(n):
        row_tiles, col_tiles = (n + 127) // 128, (n + 255) // 256
        return sum(col_tiles - rb // 2 for rb in range(row_tiles))
    launched = computing = 0
    for lo_i in range(0, rows, panel):
        ri = min(panel, rows - lo_i)
        launched += triangle(ri)
        computing += triangle(ri)
        for lo_j in range(lo_i + panel, rows, panel):
            rj = min(panel, rows - lo_j)
            launched += triangle(panel + rj)
            computing += (panel // 128) * ((rj + 255) // 256)
    return launched, computing


def phase_times(torch, eng, steps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            eng.exact_moments_device(std=True)
        torch.cuda.synchronize()
    out = {name: 0.0 for name, _ in PHASES}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        us = ev.cuda_time_total if us is None else us
        for name, keys in PHASES:
            if any(k in ev.key for k in keys):
                out[name] += us / 1000.0 / steps
    return out


def timed(torch, fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_config(name, args, log):
    import torch
    from pangenomix_b200 import pangenome_analysis as pa, sparse_utils as su, synth
    coo = load(name)
    n_genes, n = coo.shape
    df = su.LightSparseDataFrame(*synth.labels_for(n_genes, n), coo)
    eng = pa._engine_for(df)
    hp = eng.host_plan
    rows = hp.n_rows + hp.n_long
    n_pad = -(-n // 128) * 128
    work = eng.pair_workspace_bytes()
    e_rows = (work - int(eng.lib.pgx_pair_overlap_work_bytes(n, rows, 1)) + (-(-rows // 128) * 128) * n_pad) // n_pad
    panel = rows if e_rows >= -(-rows // 128) * 128 else e_rows // 2 // 256 * 256
    launched, computing = launched_tiles(rows, panel)
    res = {"config": name, "n_genes": n_genes, "n_genomes": n, "stored_rows": rows, "n_rows": hp.n_rows,
           "n_long": hp.n_long, "workspace_bytes": work, "panel_rows": panel, "tiles_launched": launched,
           "tiles_computing": computing}
    log("%s: N = %d, G = %d, stored rows %d (list %d, bitmap %d), workspace %.2f GB, panel %d rows, %d panel(s), "
        "GEMM tiles %d computing of %d launched" % (name, n, n_genes, rows, hp.n_rows, hp.n_long, work / 1e9, panel,
                                                   -(-rows // panel), computing, launched))

    for _ in range(args.warmup):
        pa.exact_pan_core_summary(df)
        pa.exact_pan_core_summary(df, std=False)
    torch.cuda.synchronize()
    res["phases_ms"] = phase_times(torch, eng, args.steps)
    log("  phases (ms, profiler device time per call): " + ", ".join("%s %.3f" % kv for kv in res["phases_ms"].items()))
    ops = 2.0 * computing * 128 * 256 * n_pad
    g = res["phases_ms"]["gemm"]
    if g > 0:
        res["gemm_tops"] = ops / (g * 1e-3) / 1e12
        res["gemm_share_of_4_5_pops"] = ops / (g * 1e-3) / INT8_DENSE_OPS
        log("  gemm: %.3g ops over the computing tiles in %.3f ms = %.0f TOPS = %.1f %% of 4.5 POPS" % (
            ops, g, res["gemm_tops"], 100 * res["gemm_share_of_4_5_pops"]))
    res["api_std_false_ms"] = timed(torch, lambda: pa.exact_pan_core_summary(df, std=False), args.steps)
    res["api_std_true_ms"] = timed(torch, lambda: pa.exact_pan_core_summary(df), args.steps)
    log("  exact_pan_core_summary (CUDA events, %d calls): std=False %.3f ms, std=True %.3f ms" % (
        args.steps, res["api_std_false_ms"], res["api_std_true_ms"]))
    out = pa.exact_pan_core_summary(df)
    res["pan_mean_at_N"] = float(out.loc["mean"].iloc[n - 1])
    res["pan_std_max"] = float(out.loc["std"].iloc[:n].max())
    res["core_std_max"] = float(out.loc["std"].iloc[n:].max())
    log("  pan mean at N %.1f (G %d), largest pan std %.3f, largest core std %.3f" % (
        res["pan_mean_at_N"], n_genes, res["pan_std_max"], res["core_std_max"]))

    if args.shared:
        for _ in range(args.warmup):
            eng.fluidity_rows_device(eng.shared_genes_device())
        torch.cuda.synchronize()
        sp = shared_phase_times(torch, eng, args.steps)
        s_ops, _ = gemm_counts(hp)
        res["shared_gemm_ms"] = sp["gemm"]
        res["shared_gemm_share_of_4_5_pops"] = s_ops / (sp["gemm"] * 1e-3) / INT8_DENSE_OPS
        log("  pgx_shared_genes gemm in the same run: %.3f ms = %.1f %% of 4.5 POPS" % (
            sp["gemm"], 100 * res["shared_gemm_share_of_4_5_pops"]))
    pa._ENGINE_CACHE.clear()
    del eng
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("out")
    ap.add_argument("--configs", default="c4,c5")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--no-shared", dest="shared", action="store_false")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_exact_rarefaction.py needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    tag = args.configs.replace(",", "_")
    lines = []

    def log(msg):
        print(msg, flush=True)
        lines.append(msg)

    info = {"card": card(), "device": torch.cuda.get_device_name()}
    log("card (name, power limit, max SM clock): %s" % info["card"])
    info["results"] = [run_config(name, args, log) for name in args.configs.split(",")]
    with open(os.path.join(args.out, "exact_%s.json" % tag), "w") as f:
        json.dump(info, f, indent=1)
    with open(os.path.join(args.out, "exact_%s.log" % tag), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
