"""Throughput of the seeded on-device rarefaction path (estimate_pan_core_summary) against the kernels alone.

    python scripts/probe_pan_core_summary.py [--configs c4,c5] [--steps 40] [--warmup 3] [--out DIR]
    torchrun --nproc_per_node 8 scripts/probe_pan_core_summary.py ...     (adds the sharded call on 8 GPUs)

Per config (C4: 10,000 permutations per step, C5: 1,000), on one GPU, all timed with CUDA events over back-to-back
steps after warm-up:
  kernels   pgx_pan_core_curves on permutations drawn beforehand (what bench.py reports as ``value``)
  gen       pgx_random_perms alone;  moments: pgx_curve_moments alone (on the curve block of a step)
  summary   PanCoreEngine.summary_device: generate -> curves -> moments per block, the whole API hot path
  api       estimate_pan_core_summary end to end (host clock, including the DataFrame), steps x perms per step
  drop-in   estimate_pan_core_size(df, 2000) (host clock; numpy's bit-exact stream, float64 table to the host)
Under torchrun every rank also runs estimate_pan_core_summary_sharded with steps x perms per step x world
permutations (host clock between barriers).  The card's name and power limit are printed with the numbers.
Writes DIR/pan_core_summary_<configs>_n<world>.json (default DIR: profiles/r03).
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

PERMS_PER_STEP = {"c1": 10000, "c2": 10000, "c4": 10000, "c5": 1000}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def load(name):
    import scipy.sparse
    from pangenomix_b200 import synth
    n_genes, n_genomes, _, seed, _ = synth.CONFIGS[name]
    cache = os.path.join(tempfile.gettempdir(), "pgx_synth_%s_%d.npy" % (name, seed))
    if not os.path.exists(cache):
        coo = synth.config_matrix(name)
        tmp = cache + ".tmp%d.npy" % os.getpid()
        np.save(tmp, np.stack([coo.row.astype(np.int32), coo.col.astype(np.int32)]))
        os.replace(tmp, cache)
    packed = np.load(cache)
    return scipy.sparse.coo_matrix((np.ones(packed.shape[1], dtype=np.int64), (packed[0], packed[1])),
                                   shape=(n_genes, n_genomes))


def timed(torch, fn, steps, warmup):
    """ms per call of fn over ``steps`` back-to-back calls, CUDA events around the whole window."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_config(name, args, rank, world, log):
    import torch
    from pangenomix_b200 import _native, distributed, engine, pangenome_analysis as pa, sparse_utils as su, synth
    coo = load(name)
    lsdf = su.LightSparseDataFrame(*synth.labels_for(*coo.shape), coo)
    eng = pa._engine_for(lsdf)
    n, p = coo.shape[1], PERMS_PER_STEP[name]
    res = {"config": name, "n_genomes": n, "n_genes": coo.shape[0], "nnz": int(coo.nnz), "perms_per_step": p,
           "steps": args.steps}
    lib = _native.load()
    perms = torch.empty((p, n), dtype=torch.int16, device=eng.device)
    curves = torch.empty((p, 2 * n), dtype=torch.int32, device=eng.device)
    mom = [torch.empty(2 * n, dtype=d, device=eng.device) for d in (torch.int64, torch.int64, torch.int32, torch.int32)]
    stream = torch.cuda.current_stream().cuda_stream
    engine.random_permutations_device(n, p, 1, out=perms)
    if rank == 0:
        ms = {
            "kernels": timed(torch, lambda: eng.curves_device(perms, out=curves), args.steps, args.warmup),
            "gen": timed(torch, lambda: engine.random_permutations_device(n, p, 1, out=perms), args.steps, args.warmup),
            "moments": timed(torch, lambda: _native.check(lib.pgx_curve_moments(
                curves.data_ptr(), p, 2 * n, *[m.data_ptr() for m in mom], 1, stream)), args.steps, args.warmup),
        }
        steps = args.steps
        eng.summary_device(p * args.warmup, 7, block=p)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.summary_device(p * steps, 7, block=p)
        e1.record()
        torch.cuda.synchronize()
        ms["summary"] = e0.elapsed_time(e1) / steps
        t = time.perf_counter()
        pa.estimate_pan_core_summary(lsdf, p * steps, seed=7)
        ms["api"] = (time.perf_counter() - t) * 1e3 / steps
        with contextlib.redirect_stdout(io.StringIO()):
            pa.estimate_pan_core_size(lsdf, 64)
            t = time.perf_counter()
            pa.estimate_pan_core_size(lsdf, 2000)
            dropin_s = time.perf_counter() - t
        res["ms_per_step"] = ms
        res["perms_per_s"] = {k: p / (v / 1e3) for k, v in ms.items()}
        res["perms_per_s"]["drop_in_2000"] = 2000 / dropin_s
        res["api_over_kernels"] = ms["kernels"] / ms["api"]
        res["summary_over_kernels"] = ms["kernels"] / ms["summary"]
        log("[%s] N=%d G=%d, %d perms/step, %d steps: kernels %.3f ms, gen %.3f ms, moments %.3f ms, summary %.3f ms, "
            "api %.3f ms per step" % (name, n, coo.shape[0], p, steps, ms["kernels"], ms["gen"], ms["moments"],
                                      ms["summary"], ms["api"]))
        log("[%s] perms/s: kernels %.0f, summary %.0f (%.1f %%), api %.0f (%.1f %% of kernels), drop-in "
            "estimate_pan_core_size(2000) %.0f" % (name, res["perms_per_s"]["kernels"], res["perms_per_s"]["summary"],
                                                     100 * res["summary_over_kernels"], res["perms_per_s"]["api"],
                                                     100 * res["api_over_kernels"], res["perms_per_s"]["drop_in_2000"]))
    if world > 1:
        import torch.distributed as dist
        total = p * args.steps * world
        distributed.estimate_pan_core_summary_sharded(lsdf, p * world, seed=7)      # warm-up
        dist.barrier()
        torch.cuda.synchronize()
        t = time.perf_counter()
        distributed.estimate_pan_core_summary_sharded(lsdf, total, seed=7)
        dist.barrier()
        sharded_s = time.perf_counter() - t
        res["sharded"] = {"world": world, "perms": total, "seconds": sharded_s, "perms_per_s": total / sharded_s}
        if rank == 0:
            log("[%s] sharded over %d GPUs: %d perms in %.3f s = %.0f perms/s" % (name, world, total, sharded_s,
                                                                              total / sharded_s))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", default="c4,c5")
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r03"))
    args = ap.parse_args()
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def log(msg):
        if rank == 0:
            print(msg, flush=True)

    info = {"card": card(), "torch_device": torch.cuda.get_device_name(local), "world": world, "results": []}
    log("card (name, power limit, max SM clock): %s" % info["card"])
    for name in args.configs.split(","):
        info["results"].append(run_config(name.strip(), args, rank, world, log))
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        path = os.path.join(args.out, "pan_core_summary_%s_n%d.json" % (args.configs.replace(",", "_"), world))
        with open(path, "w") as f:
            json.dump(info, f, indent=1)
        log("wrote %s" % path)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
