#!/usr/bin/env python
"""Generates tests/golden/*.npz by running the LIVE reference (/root/reference).

Run in the build container only (the reference does not exist on the GPU box):

    python tests/golden/make_golden.py            # the round-1 fixtures
    python tests/golden/make_golden.py --big      # the full-size fixtures of round 2 (C2, C4, C3; ~6 min)
    python tests/golden/make_golden.py --betabin  # beta-binomial core estimate, Monte-Carlo KS, gene occurrence
    python tests/golden/make_golden.py --c5       # one permutation of config C5 at full size (tens of minutes)
    python tests/golden/make_golden.py --c3-whole # the reference's Bernoulli fit on the whole table, 40,000 x 400 (minutes)

The reference has no tests or golden vectors of its own (SURVEY.md section 4), so
these fixtures -- outputs of the unmodified reference functions under a fixed
``np.random.seed`` -- are what pins the oracle and the CUDA path.  The reference
imports ``statsmodels`` at pangenome_analysis.py:18 but only uses it at :380 (off the
hot path); it is absent from this image, so an empty module is registered in
``sys.modules`` before the import.  Nothing else is patched.

Versions at generation time are recorded in tests/golden/MANIFEST.json.
"""
import contextlib
import hashlib
import io
import json
import os
import sys
import types
import warnings

import numpy as np
import pandas as pd
import scipy
import scipy.sparse

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True
sys.path.insert(0, "/root/reference")
for name in ("statsmodels", "statsmodels.stats", "statsmodels.stats.stattools"):
    sys.modules.setdefault(name, types.ModuleType(name))
sys.modules["statsmodels"].stats = sys.modules["statsmodels.stats"]
sys.modules["statsmodels.stats"].stattools = sys.modules["statsmodels.stats.stattools"]
# the one statsmodels function the reference calls (pangenome_analysis.py:380), by its textbook definition
sys.modules["statsmodels.stats.stattools"].durbin_watson = \
    lambda resids: float(np.sum(np.diff(resids) ** 2) / np.sum(np.asarray(resids) ** 2))

import pangenomix.pangenome_analysis as ref_pa  # noqa: E402  (the reference)
import pangenomix.sparse_utils as ref_su  # noqa: E402

from pangenomix_b200 import synth  # noqa: E402


def quiet(fn, *args, **kwargs):
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fn(*args, **kwargs)


def matrix_digest(coo):
    coo = scipy.sparse.coo_matrix(coo)
    order = np.lexsort((coo.col, coo.row))
    h = hashlib.sha256()
    h.update(np.asarray(coo.shape, dtype=np.int64).tobytes())
    h.update(coo.row[order].astype(np.int32).tobytes())
    h.update(coo.col[order].astype(np.int32).tobytes())
    h.update(coo.data[order].astype(np.int64).tobytes())
    return h.hexdigest()


def lsdf_of(coo):
    index, columns = synth.labels_for(*coo.shape)
    return ref_su.LightSparseDataFrame(index, columns, coo)


def run_curves(coo, seed, num_iter):
    """Reference curves + the permutations the reference consumed for them."""
    np.random.seed(seed)
    df = quiet(ref_pa.estimate_pan_core_size, lsdf_of(coo), num_iter)
    np.random.seed(seed)
    n = coo.shape[1]
    perms = np.empty((num_iter, n), dtype=np.int64)
    for i in range(num_iter):
        a = np.arange(n)
        np.random.shuffle(a)
        perms[i] = a
    assert df.values.dtype == np.float64
    assert list(df.index) == ["Iter%d" % (i + 1) for i in range(num_iter)]
    assert list(df.columns) == ["Pan%d" % (i + 1) for i in range(n)] + \
        ["Core%d" % (i + 1) for i in range(n)]
    return df, perms


def save_curve_case(name, coo, seed, num_iter, store_matrix=True, heaps=False):
    coo = scipy.sparse.coo_matrix(coo)
    df, perms = run_curves(coo, seed, num_iter)
    out = {
        "shape": np.asarray(coo.shape, dtype=np.int64),
        "seed": np.int64(seed),
        "num_iter": np.int64(num_iter),
        # uint16 where the counts fit (lossless, asserted below): keeps C2's 1,000 curves under 1 MB
        "curves": df.values.astype(np.uint16 if df.values.max() <= 65535 else np.int32),
        "digest": np.array(matrix_digest(coo)),
    }
    assert np.array_equal(out["curves"].astype(np.float64), df.values)
    if store_matrix:
        out["row"] = coo.row.astype(np.int32)
        out["col"] = coo.col.astype(np.int32)
        out["data"] = coo.data.astype(np.int64)
    if perms.shape[1] <= 64:
        out["perms"] = perms.astype(np.int32)
    if heaps:
        mean_df = pd.DataFrame([df.mean()], columns=df.columns)   # plot.py:8-11
        out["mean"] = mean_df.values[0]
        out["heaps_mean"] = quiet(ref_pa.fit_heaps_by_iteration, mean_df).values[0]
        out["heaps_iter"] = quiet(ref_pa.fit_heaps_by_iteration, df.iloc[:min(num_iter, 8)]).values
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("wrote", name, coo.shape, "nnz", coo.nnz, "iters", num_iter)


def edge_matrix():
    """500 x 37 with all-present, empty, single-present, single-absent and duplicate rows."""
    rng = np.random.RandomState(99)
    x = (rng.random_sample((500, 37)) < rng.beta(0.4, 0.4, size=(500, 1))).astype(np.int64)
    x[0:10] = 1                       # all-present
    x[10:20] = 0                      # empty
    x[20:40] = 0
    x[np.arange(20, 40), rng.randint(37, size=20)] = 1      # singletons
    x[40:60] = 1
    x[np.arange(40, 60), rng.randint(37, size=20)] = 0      # single-absent
    x[60:70] = x[70:80]               # identical rows
    return scipy.sparse.coo_matrix(x)


def big_cases(manifest):
    """Round-2 additions: live-reference fixtures at the sizes the performance claims are made on.

    c2_40000x400      config C2 in full: all of its 1,000 permutations (the reference needs 0.1 s each), their mean,
                      the Heaps fit on the mean
    c4_200000x10000   config C4 in full, 16 of its 10,000 permutations (the reference needs ~9 s each)
    bernoulli_c3_4000x400  config C3 (candidate-core size): the whole L-BFGS-B fit of the reference (~10 s)
    The matrices are regenerated by pangenomix_b200.synth in the tests and checked against the stored digest.
    """
    c2 = synth.config_matrix("c2")
    save_curve_case("c2_40000x400", c2, 12345, 1000, store_matrix=False, heaps=True)
    c4 = synth.config_matrix("c4")
    save_curve_case("c4_200000x10000", c4, 12345, 16, store_matrix=False, heaps=True)

    x, p_true, q_true = synth.bernoulli_grid_matrix(4000, 400, seed=3)
    n_genes, n_genomes = x.shape
    index, columns = synth.labels_for(n_genes, n_genomes)
    dense = pd.DataFrame(x, index=index, columns=columns)
    import time
    t = time.time()
    df_opt, res = quiet(ref_pa.compute_bernoulli_grid_core_genome, dense)
    fit_seconds = time.time() - t
    ll = ref_pa.__dict__["__bernoulli_grid_loglikelihood__"]
    grad = ref_pa.__dict__["__bernoulli_grid_loglikelihood_gradient__"]
    init = df_opt["initial"].values[1:]
    opt = df_opt["optimum"].values[1:]
    np.savez_compressed(
        os.path.join(HERE, "bernoulli_c3_4000x400.npz"),
        shape=np.asarray(x.shape, dtype=np.int64), x_digest=np.array(hashlib.sha256(x.astype(np.uint8).tobytes()).hexdigest()),
        fit_initial=df_opt["initial"].values, fit_optimum=df_opt["optimum"].values,
        fit_x=res.x, fit_fun=np.float64(res.fun), fit_nit=np.int64(res.nit), fit_nfev=np.int64(res.nfev),
        fit_message=np.array(str(res.message)), fit_seconds=np.float64(fit_seconds),
        ll_init=np.float64(ll(x, init[:n_genes], init[n_genes:])), grad_init=grad(x, init[:n_genes], init[n_genes:]),
        ll_opt=np.float64(ll(x, opt[:n_genes], opt[n_genes:])), grad_opt=grad(x, opt[:n_genes], opt[n_genes:]))
    manifest["bernoulli_c3_4000x400_reference_fit_seconds"] = fit_seconds
    print("wrote bernoulli_c3_4000x400: init LL", df_opt["initial"].values[0], "opt LL", -res.fun, "nit", res.nit,
          "nfev", res.nfev, "%.1fs" % fit_seconds)


def betabin_cases(manifest):
    """Round-2 additions for SURVEY.md section 8(f) row 4: compute_beta_binomial_core_genome (pangenome_analysis.py:
    295-400) and its Monte-Carlo KS test (:457-482) as the live reference computes them, together with every call of
    ks_montecarlo_bbn they make (arguments and results recorded by a pass-through wrapper) and the state of the
    global numpy RNG afterwards.  statsmodels is absent from the image: durbin_watson is the textbook formula."""
    calls = []
    original = ref_pa.ks_montecarlo_bbn

    def recorder(ycounts, n, a, b, iterations=100, sim_limit=1000):
        out = original(ycounts, n, a, b, iterations=iterations, sim_limit=sim_limit)
        calls.append({"x": np.asarray(ycounts.index, dtype=np.int64), "y": np.asarray(ycounts.values, dtype=np.int64),
                      "n": int(n), "a": float(a), "b": float(b), "iterations": int(iterations),
                      "sim_limit": int(sim_limit), "pvalue": float(out[0]), "ks_stat": float(out[1]),
                      "ks_sim": np.asarray(out[2], dtype=np.float64)})
        return out

    def run(name, df_genes, df_counts, num_points, ks_iter, seed, extra=None):
        del calls[:]
        ref_pa.ks_montecarlo_bbn = recorder
        try:
            np.random.seed(seed)
            out = quiet(ref_pa.compute_beta_binomial_core_genome, df_genes, df_counts=df_counts,
                        num_points=num_points, ks_iter=ks_iter)
        finally:
            ref_pa.ks_montecarlo_bbn = original
        state = np.random.get_state()
        table = out.to_frame().T if isinstance(out, pd.Series) else out
        points = [num_points] if isinstance(num_points, int) else list(num_points)
        store = {"num_points": np.asarray(points, dtype=np.int64), "single": np.bool_(isinstance(out, pd.Series)),
                 "ks_iter": np.int64(ks_iter), "seed": np.int64(seed), "columns": np.array(list(table.columns)),
                 "result": table.values.astype(np.float64), "n_ks_calls": np.int64(len(calls)),
                 "rng_key_after": np.asarray(state[1], dtype=np.uint32), "rng_pos_after": np.int64(state[2])}
        if df_counts is not None:
            store["counts_index"] = np.asarray(df_counts.index, dtype=np.int64)
            store["counts_values"] = np.asarray(df_counts.values, dtype=np.int64)
        for i, call in enumerate(calls):
            for key, value in call.items():
                store["ks%d_%s" % (i, key)] = np.asarray(value)
        store.update(extra or {})
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **store)
        print("wrote", name, "points", points, "ks calls", len(calls))
        print(table.to_string())

    f, c = synth.core_miss_spectrum()
    run("betabin_spectrum300", None, pd.Series(c, index=f), [10, 15, 25, 40], 200, 3)
    f, c = synth.core_miss_spectrum(n_genomes=2000, n_core=40000, a=0.4, b=300.0, n_accessory=20000, seed=5)
    run("betabin_spectrum2000", None, pd.Series(c, index=f), [15, 25, 40], 100, 4)
    run("betabin_spectrum2000_single", None, pd.Series(c, index=f), 25, 60, 9)
    # config C1's own spectrum (the reference's fit is poor there: p = 0)
    c1 = synth.config_matrix("c1")
    spectrum = np.bincount(np.bincount(c1.row, minlength=c1.shape[0]), minlength=c1.shape[1] + 1)
    keep = np.flatnonzero(spectrum[1:]) + 1
    run("betabin_c1", None, pd.Series(spectrum[keep].astype(np.int64), index=keep.astype(np.int64)), 10, 50, 12345)
    # the df_genes path (:352-355): the spectrum is a collections.Counter of the row sums, i.e. ordered by FIRST
    # APPEARANCE of each frequency among the rows, and ``iloc[-n_points:]`` (:364) takes the last of that order.
    # (a) rows sorted by ascending frequency, so that the order is the sorted one; (b) rows as generated.
    f, c = synth.core_miss_spectrum(n_genomes=60, n_core=3000, a=0.7, b=25.0, n_accessory=600, seed=21)
    x = synth.table_with_frequencies(np.repeat(f, c), 60, seed=22)
    index, columns = synth.labels_for(*x.shape)
    dfs = pd.DataFrame.sparse.from_spmatrix(x.tocsc(), index=index, columns=columns)
    run("betabin_table_sorted_3600x60", dfs, None, [10, 20], 80, 6,
        extra={"row": x.row.astype(np.int32), "col": x.col.astype(np.int32), "shape": np.asarray(x.shape, dtype=np.int64)})
    small = scipy.sparse.coo_matrix(synth.bernoulli_matrix(800, 50, 450, seed=7))
    index, columns = synth.labels_for(*small.shape)
    dfs = pd.DataFrame.sparse.from_spmatrix(small.tocsc(), index=index, columns=columns)
    run("betabin_table_unsorted_800x50", dfs, None, 10, 40, 6,
        extra={"row": small.row.astype(np.int32), "col": small.col.astype(np.int32),
               "shape": np.asarray(small.shape, dtype=np.int64)})
    # count_gene_occurence (core_genome.py:127-155) on the same table, read from the .npz the reference writes
    import tempfile
    bio = types.ModuleType("Bio")                 # core_genome.py:3 imports Bio.SeqIO (absent here, unused by the function)
    bio.SeqIO = types.ModuleType("Bio.SeqIO")
    sys.modules.setdefault("Bio", bio)
    sys.modules.setdefault("Bio.SeqIO", bio.SeqIO)
    import pangenomix.core_genome as ref_cg
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "t.npz")
        lsdf_of(small).to_npz(path)
        occ = quiet(ref_cg.count_gene_occurence, path)
    np.savez_compressed(os.path.join(HERE, "gene_occurence_800x50.npz"), gene_index=occ["gene_index"].values,
                        count=occ["count"].values, columns=np.array(list(occ.columns)),
                        row=small.row.astype(np.int32), col=small.col.astype(np.int32),
                        shape=np.asarray(small.shape, dtype=np.int64))
    print("wrote gene_occurence_800x50", occ.shape, occ.dtypes.to_dict())


def bernoulli_whole_table_case(manifest):
    """Config C3 on the whole table (40,000 genes x 400 genomes, README.md:199-211): the reference's full L-BFGS-B fit
    (minutes), its LL and gradient at the start point and at its optimum."""
    import time
    x, _, _ = synth.bernoulli_grid_matrix(40000, 400, seed=3)
    n_genes, n_genomes = x.shape
    index, columns = synth.labels_for(n_genes, n_genomes)
    dense = pd.DataFrame(x, index=index, columns=columns)
    t = time.time()
    df_opt, res = quiet(ref_pa.compute_bernoulli_grid_core_genome, dense)
    fit_seconds = time.time() - t
    ll = ref_pa.__dict__["__bernoulli_grid_loglikelihood__"]
    grad = ref_pa.__dict__["__bernoulli_grid_loglikelihood_gradient__"]
    init = df_opt["initial"].values[1:]
    opt = df_opt["optimum"].values[1:]
    np.savez_compressed(
        os.path.join(HERE, "bernoulli_c3_40000x400.npz"),
        shape=np.asarray(x.shape, dtype=np.int64), x_digest=np.array(hashlib.sha256(x.astype(np.uint8).tobytes()).hexdigest()),
        fit_ll_initial=np.float64(df_opt["initial"].values[0]), fit_x=res.x, fit_fun=np.float64(res.fun),
        fit_nit=np.int64(res.nit), fit_nfev=np.int64(res.nfev), fit_message=np.array(str(res.message)),
        fit_seconds=np.float64(fit_seconds),
        ll_init=np.float64(ll(x, init[:n_genes], init[n_genes:])), grad_init=grad(x, init[:n_genes], init[n_genes:]),
        ll_opt=np.float64(ll(x, opt[:n_genes], opt[n_genes:])), grad_opt=grad(x, opt[:n_genes], opt[n_genes:]))
    manifest["bernoulli_c3_40000x400_reference_fit_seconds"] = fit_seconds
    print("wrote bernoulli_c3_40000x400: init LL", df_opt["initial"].values[0], "opt LL", -res.fun, "nit", res.nit,
          "nfev", res.nfev, "%.1fs" % fit_seconds)


def c5_case(manifest):
    """Config C5 at full size (2,000,000 alleles x 50,000 genomes, nnz 2.0e8): ONE permutation through the live
    reference (about 50,000 dense passes over 2 M counters: tens of minutes on the build host)."""
    import time
    c5 = synth.config_matrix("c5")
    t = time.time()
    save_curve_case("c5_2000000x50000", c5, 12345, 1, store_matrix=False, heaps=False)
    manifest["c5_2000000x50000_reference_seconds_per_permutation"] = time.time() - t


def main():
    if "--c3-whole" in sys.argv:
        path = os.path.join(HERE, "MANIFEST.json")
        with open(path) as f:
            manifest = json.load(f)
        bernoulli_whole_table_case(manifest)
        with open(path, "w") as f:
            json.dump(manifest, f, indent=1, sort_keys=True)
        return
    if "--c5" in sys.argv:
        path = os.path.join(HERE, "MANIFEST.json")
        with open(path) as f:
            manifest = json.load(f)
        c5_case(manifest)
        with open(path, "w") as f:
            json.dump(manifest, f, indent=1, sort_keys=True)
        return
    if "--betabin" in sys.argv:
        path = os.path.join(HERE, "MANIFEST.json")
        with open(path) as f:
            manifest = json.load(f)
        betabin_cases(manifest)
        manifest["betabin"] = "statsmodels absent: durbin_watson = sum(diff(r)^2) / sum(r^2)"
        with open(path, "w") as f:
            json.dump(manifest, f, indent=1, sort_keys=True)
        return
    if "--big" in sys.argv:
        path = os.path.join(HERE, "MANIFEST.json")
        with open(path) as f:
            manifest = json.load(f)
        big_cases(manifest)
        with open(path, "w") as f:
            json.dump(manifest, f, indent=1, sort_keys=True)
        return
    manifest = {
        "numpy": np.__version__, "scipy": scipy.__version__, "pandas": pd.__version__,
        "python": sys.version.split()[0],
        "reference": "/root/reference/pangenomix (AnnaLew/pangenomix, unmodified; statsmodels stubbed)",
    }
    # 1. the survey's known-answer matrix
    kat = np.array([[1, 1, 1, 1, 1], [1, 0, 1, 1, 1], [0, 0, 1, 0, 0],
                    [1, 1, 0, 0, 0], [0, 0, 0, 0, 1], [0, 1, 1, 0, 1]], dtype=np.int64)
    save_curve_case("kat_6x5", scipy.sparse.coo_matrix(kat), 12345, 3, heaps=True)
    # 2. small synthetic, two seeds
    small = synth.bernoulli_matrix(800, 50, 450, seed=7)
    save_curve_case("synth_800x50_s0", small, 0, 10, heaps=True)
    save_curve_case("synth_800x50_s1", small, 1, 10)
    # 3. edge rows
    save_curve_case("edge_500x37", edge_matrix(), 1, 20)
    # 4. tiny shapes
    for n in (1, 2, 3, 4):
        rng = np.random.RandomState(n)
        x = (rng.random_sample((40, n)) < 0.5).astype(np.int64)
        save_curve_case("tiny_40x%d" % n, scipy.sparse.coo_matrix(x), 5, 6)
    # 5. config C1 in full (matrix regenerated by synth in the tests; digest stored)
    c1 = synth.config_matrix("c1")
    save_curve_case("c1_8000x50", c1, 12345, 100, store_matrix=False, heaps=True)
    # 6. a 4000 x 400 table shaped like a slice of C2
    c2s = synth.bernoulli_matrix(4000, 400, 450, seed=20242)
    save_curve_case("c2slice_4000x400", c2s, 12345, 5, store_matrix=False, heaps=True)
    # 7. duplicates in the COO are summed by .tocsr() (:75): pan unaffected, core changes
    dup = scipy.sparse.coo_matrix(
        (np.ones(9, dtype=np.int64),
         (np.array([0, 0, 0, 1, 1, 2, 2, 2, 2]), np.array([0, 0, 1, 1, 2, 0, 1, 2, 3]))),
        shape=(3, 4))
    df, perms = run_curves(dup, 3, 4)
    np.savez_compressed(os.path.join(HERE, "dup_3x4.npz"), row=dup.row.astype(np.int32),
                        col=dup.col.astype(np.int32), data=dup.data.astype(np.int64),
                        shape=np.asarray(dup.shape, dtype=np.int64), perms=perms.astype(np.int32),
                        curves=df.values.astype(np.int32), seed=np.int64(3), num_iter=np.int64(4))
    print("wrote dup_3x4")

    # 8. Bernoulli grid: likelihood, gradient, full fit
    x, p_true, q_true = synth.bernoulli_grid_matrix(300, 40, seed=3)
    n_genes, n_genomes = x.shape
    lo, hi = 0.8, 0.99999999
    p0 = np.clip(x.sum(axis=1) / float(n_genomes), lo, hi)
    q0 = np.clip(0.9999 * np.ones(n_genomes), lo, hi)
    rng = np.random.RandomState(11)
    p1 = rng.uniform(lo, hi, size=n_genes)
    q1 = rng.uniform(lo, hi, size=n_genomes)
    ll = ref_pa.__dict__["__bernoulli_grid_loglikelihood__"]
    grad = ref_pa.__dict__["__bernoulli_grid_loglikelihood_gradient__"]
    index, columns = synth.labels_for(n_genes, n_genomes)
    dense = pd.DataFrame(x, index=index, columns=columns)
    df_opt, res = quiet(ref_pa.compute_bernoulli_grid_core_genome, dense)
    assert list(df_opt.columns) == ["initial", "optimum"]
    assert list(df_opt.index) == ["Loglikelihood"] + ["p_" + s for s in index] + ["q_" + s for s in columns]
    x2 = kat[:2].astype(np.float64)
    np.savez_compressed(
        os.path.join(HERE, "bernoulli_300x40.npz"),
        x=x.astype(np.uint8), p0=p0, q0=q0, p1=p1, q1=q1,
        ll0=np.float64(ll(x, p0, q0)), grad0=grad(x, p0, q0),
        ll1=np.float64(ll(x, p1, q1)), grad1=grad(x, p1, q1),
        fit_initial=df_opt["initial"].values, fit_optimum=df_opt["optimum"].values,
        fit_x=res.x, fit_fun=np.float64(res.fun), fit_nit=np.int64(res.nit),
        fit_nfev=np.int64(res.nfev), fit_message=np.array(str(res.message)),
        kat_x=x2, kat_p=np.array([0.99999999, 0.8]), kat_q=0.9999 * np.ones(5),
        kat_ll=np.float64(ll(x2, np.array([0.99999999, 0.8]), 0.9999 * np.ones(5))),
        kat_grad=grad(x2, np.array([0.99999999, 0.8]), 0.9999 * np.ones(5)))
    print("wrote bernoulli_300x40: init LL", df_opt["initial"].values[0], "opt LL", -res.fun,
          "nit", res.nit)

    # 9. LSDF .npz round trip as the reference writes it (sparse_utils.py:295-314)
    tmp = os.path.join(HERE, "lsdf_small.npz")
    lsdf = lsdf_of(small)
    lsdf.to_npz(tmp)
    back = ref_su.read_lsdf(tmp)
    assert (back.data != lsdf.data).nnz == 0
    manifest["lsdf_small_row_sums_head"] = [int(v) for v in lsdf.sum(axis="index")[:8]]
    manifest["lsdf_small_col_sums_head"] = [int(v) for v in lsdf.sum(axis="columns")[:8]]
    print("wrote lsdf_small.npz (+ .labels.txt) with the reference's own writer")

    with open(os.path.join(HERE, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
