"""Drop-in for the analysis hot path of /root/reference/pangenomix/pangenome_analysis.py.

Same function names, arguments, printed lines, return types, labels and dtypes as the
reference; the work is done by libpgx_b200 on a B200:

* ``estimate_pan_core_size``  (:51-98)  -> PanCoreEngine (min-rank kernels, bit-exact)
* ``fit_heaps_by_iteration``  (:24-48)  -> unchanged host scipy ``curve_fit`` on the curves
* ``compute_bernoulli_grid_core_genome`` (:101-166) -> scipy L-BFGS-B on the host driving
  the fp64 likelihood/gradient kernel (BernoulliGrid)

* ``compute_beta_binomial_core_genome`` (:295-400), ``ks_montecarlo_bbn`` (:457-482) -> gene-frequency spectrum
  counted on the GPU, scipy Nelder-Mead / Shapiro-Wilk on the host as in the reference, and the Monte-Carlo KS
  simulation on the GPU (pgx_ks_montecarlo_host), consuming the global numpy RNG exactly as ``np.random.choice`` does

Extension beside the drop-in: ``estimate_pan_core_summary`` -- mean / std / min / max of the pan/core curves over
genome orders drawn on the GPU from a seeded counter-based stream (not numpy's), reduced on the GPU;
``shared_gene_counts`` (genome x genome shared genes, X^T X on the tensor cores) and ``compute_genomic_fluidity``;
``exact_pan_core_summary`` -- the exact mean and std of the pan/core curves over ALL genome orders, without sampling
(gene-pair overlap histograms counted on the tensor cores).

Not provided (out of scope, SURVEY.md section 2): the coordinate-descent variant the
reference marks "DON'T USE THIS" and the mlst wrapper.
"""
from __future__ import print_function

import math
import weakref

import collections

import numpy as np
import pandas as pd
import scipy.optimize
import scipy.stats
from scipy.special import betaln

from .engine import BernoulliGrid, PanCoreEngine

_ENGINE_CACHE = weakref.WeakKeyDictionary()


def _fingerprint(data):
    """Cheap identity of a COO table: the arrays it is made of (address, length) plus a strided sample of their
    content (at most 4,096 entries each), so that an in-place edit of ``data.row / .col / .data`` is noticed with
    high probability without reading the whole table on every call (the reference re-reads it every time,
    pangenome_analysis.py:74-75).  Tables should still be treated as immutable once they have been rarefied."""
    parts = [tuple(data.shape), int(getattr(data, "nnz", 0)), getattr(data, "format", None)]
    for name in ("row", "col", "data", "indices", "indptr"):
        arr = getattr(data, name, None)
        if isinstance(arr, np.ndarray):
            step = max(1, arr.shape[0] // 4096)
            sample = np.ascontiguousarray(arr[::step])
            parts.append((name, arr.__array_interface__["data"][0], arr.shape[0], str(arr.dtype), hash(sample.tobytes())))
    return tuple(parts)


def _engine_for(df_genes, device=None):
    """One uploaded matrix per LSDF object ("uploaded once"); re-planned if ``.data`` is replaced or (as far as the
    sampled fingerprint sees) edited in place."""
    try:
        cached = _ENGINE_CACHE.get(df_genes)
    except TypeError:
        cached = None
    mark = _fingerprint(df_genes.data)
    if cached is not None and cached[0] is df_genes.data and cached[2] == mark and \
            (device is None or str(cached[1].device) == str(device)):
        return cached[1]
    engine = PanCoreEngine(df_genes.data, device=device)
    try:
        _ENGINE_CACHE[df_genes] = (df_genes.data, engine, mark)
    except TypeError:
        pass
    return engine


_LABEL_CACHE = {}


def _labels(prefixes, count):
    """pd.Index of prefix1..prefixN for every prefix in turn, exactly what pandas makes of the reference's label
    lists (pangenome_analysis.py:93-97).  The label data is immutable, so it is shared between calls: building
    the 20,000 column labels of a 10,000-genome table costs more than rarefying 500 permutations."""
    key = (prefixes, int(count))
    index = _LABEL_CACHE.get(key)
    if index is None:
        if len(_LABEL_CACHE) >= 16:
            _LABEL_CACHE.pop(next(iter(_LABEL_CACHE)))
        index = pd.Index([prefix + str(x) for prefix in prefixes for x in range(1, int(count) + 1)])
        _LABEL_CACHE[key] = index
    return index.copy(deep=False)          # a new Index object over the shared labels (its .name stays private)


def fit_heaps_by_iteration(df_pan_core):
    '''
    Fits Heaps Law (PG size = kappa * genomes^alpha) to the Pan half of every row of a
    table produced by estimate_pan_core_size() (or of its mean row) and returns a
    DataFrame with columns alpha, kappa indexed like the input rows.
    '''
    pan = df_pan_core.iloc[:, :int(df_pan_core.shape[1] / 2)].T      # genomes x rows
    fits = {}
    for pos, label in enumerate(pan.columns):
        alpha, kappa = __fit_heaps_single__(pan.iloc[:, pos])
        fits[label] = {'alpha': alpha, 'kappa': kappa}
    return pd.DataFrame.from_dict(fits, orient='index').reindex(pan.columns)


def fit_heaps_by_iteration_gpu(df_pan_core, device=None):
    '''
    Same table as fit_heaps_by_iteration() -- one Heaps Law fit (alpha, kappa) per row of a pan/core
    table -- computed for all rows at once on the GPU (libpgx pgx_heaps_fit: Levenberg-Marquardt with
    the reference's start point, run to fp64 convergence).  Agrees with the scipy fits of
    fit_heaps_by_iteration() to better than 5e-6 relative (scipy's own stopping tolerance); meant for fitting every iteration of a
    large table, where thousands of scipy.optimize.curve_fit calls take minutes.
    '''
    from .engine import _require_cuda, _torch, fit_heaps_device
    torch = _torch()
    dev = _require_cuda(device)
    n_points = int(df_pan_core.shape[1] / 2)
    pan = np.ascontiguousarray(df_pan_core.values[:, :n_points], dtype=np.float64)
    fit, info = fit_heaps_device(torch.from_numpy(pan).to(dev), n_points=n_points)
    fit, info = fit.cpu().numpy(), info.cpu().numpy()
    if np.any(info < 0):
        raise RuntimeError("Heaps fit did not converge for rows %s" % np.flatnonzero(info < 0)[:8].tolist())
    return pd.DataFrame(fit, index=df_pan_core.index, columns=['alpha', 'kappa'])


def __fit_heaps_single__(df_freqs):
    ''' One Heaps Law fit; start point alpha = 0.5, kappa = min(y) as in the reference (:45). '''
    y = df_freqs.values
    x = np.arange(1, y.shape[0] + 1)
    popt, _ = scipy.optimize.curve_fit(
        lambda x, alpha, kappa: kappa * np.power(x, alpha), x, y, p0=[0.5, float(min(y))])
    return popt


def estimate_pan_core_size(df_genes, num_iter, log_batch=-1, device=None):
    '''
    Computes pan/core genome size curves for many randomizations of genome order.

    Parameters
    ----------
    df_genes : LightSparseDataFrame
        Sparse binary gene x genome table (anything with .shape and a scipy .data)
    num_iter : int
        Number of randomizations; each consumes one np.arange + np.random.shuffle from
        the global numpy RNG, exactly like the reference (:84-85).
    log_batch : int
        Prints progress every log_batch runs, or silent if negative (default -1)
    device : optional CUDA device (extension; default: current device)

    Returns
    -------
    df_pan_core : pd.DataFrame
        float64, iterations Iter1.. as index, columns Pan1..PanN, Core1..CoreN.
    '''
    num_genes, num_strains = df_genes.shape
    print('Converting DataFrame to matrix...')
    engine = _engine_for(df_genes, device)
    print('Generating pan/core curves from shuffled strains')
    curves = engine.estimate(num_iter, log_batch=log_batch)

    # labels of :93-95; the curves are a fresh array nobody else holds: wrap it instead of copying it
    # (pandas 3 copies by default)
    return pd.DataFrame(curves, index=_labels(('Iter',), num_iter),
                        columns=_labels(('Pan', 'Core'), num_strains), copy=False)


def estimate_pan_core_summary(df_genes, num_iter, seed=0, device=None):
    '''
    Mean, spread and range of the pan/core curves over ``num_iter`` random genome orders, computed without
    building the (num_iter, 2N) table: genome orders are drawn on the GPU from a seeded counter-based stream
    (pgx_random_perms; permutation i is a function of (seed, i) alone), rarefied there and reduced there to exact
    integer moments.  Only 4 x 2N numbers come back to the host.

    Unlike estimate_pan_core_size() this does not replay numpy's shuffles: it leaves ``np.random`` untouched and
    the orders it uses are not the reference's.  It prints nothing.

    Parameters
    ----------
    df_genes : LightSparseDataFrame
        Sparse binary gene x genome table (anything with .shape and a scipy .data)
    num_iter : int
        Number of random genome orders (>= 1)
    seed : int
        Seed of the stream, 0 <= seed < 2^64
    device : optional CUDA device (default: current device)

    Returns
    -------
    df_stats : pd.DataFrame
        float64, index ['mean', 'std', 'min', 'max'], columns Pan1..PanN, Core1..CoreN.  ``mean`` equals
        plot.calculate_mean() of the full table of the same orders bit for bit; ``std`` has ddof=1 as pandas
        (NaN for num_iter == 1, exactly 0 where every order gives the same value).  ``df_stats.loc[['mean']]``
        can be passed to fit_heaps_by_iteration() / fit_heaps_by_iteration_gpu().
    '''
    num_iter = int(num_iter)
    if num_iter < 1:
        raise ValueError("num_iter must be at least 1")
    _, num_strains = df_genes.shape
    engine = _engine_for(df_genes, device)
    return summary_frame(engine.summary(num_iter, seed), num_strains)


def exact_pan_core_summary(df_genes, std=True, device=None):
    '''
    Exact mean and standard deviation of the pan/core curves over ALL orders of the genomes, without sampling: the
    quantities estimate_pan_core_summary() estimates.  The first k genomes of a random order are a random k-subset,
    so with rho(v, k) = C(v, k) / C(N, k), E[core_k] = sum over genes of rho(m_g, k) and E[pan_k] = G - sum over genes
    of rho(N - m_g, k) (Mao's tau, Colwell, Mao & Chang 2004).  The variances add the pairs of genes: how many genomes
    each pair shares and how many lack both, counted on the GPU from the table's plan (shared with
    estimate_pan_core_size / estimate_pan_core_summary), the dense part as an 8-bit integer matrix product on the
    tensor cores.  The result is deterministic: no seed, no sampling noise.  Prints nothing and leaves ``np.random``
    untouched.

    Parameters
    ----------
    df_genes : LightSparseDataFrame
        Sparse binary gene x genome table (anything with .shape and a scipy .data)
    std : bool
        Also compute the std (default).  False computes the means only, which need just the gene-frequency spectrum.
    device : optional CUDA device (default: current device)

    Returns
    -------
    df_stats : pd.DataFrame
        float64, index ['mean', 'std'] (['mean'] with std=False), columns Pan1..PanN, Core1..CoreN.  ``std`` is the
        exact standard deviation over the orders of these N genomes, sqrt(max(Var, 0)); exactly 0 at k = N.
        ``df_stats.loc[['mean']]`` can be passed to fit_heaps_by_iteration() / fit_heaps_by_iteration_gpu().
    '''
    _, num_strains = df_genes.shape
    engine = _engine_for(df_genes, device)
    moments = engine.exact_moments_device(std=std).cpu().numpy()
    rows = [np.concatenate([moments[0], moments[2]])]
    if std:
        rows.append(np.sqrt(np.maximum(np.concatenate([moments[1], moments[3]]), 0.0)))
    return pd.DataFrame(np.vstack(rows), index=['mean', 'std'] if std else ['mean'],
                        columns=_labels(('Pan', 'Core'), num_strains), copy=False)


def summary_frame(moments, num_strains):
    """The DataFrame of estimate_pan_core_summary() from exact integer moments (engine.CurveMoments)."""
    n = int(moments.n)
    total = np.asarray(moments.sum, dtype=np.int64)
    mean = total.astype(np.float64) / n                     # sums below 2^53 convert exactly: pandas' mean
    if n > 1:
        # n * sum(x^2) - sum(x)^2 in Python integers, divided once: the correctly rounded ddof=1 variance
        num = np.asarray(moments.sumsq, dtype=np.uint64).astype(object) * n - total.astype(object) ** 2
        std = np.sqrt(np.array(num / (n * (n - 1)), dtype=np.float64))
    else:
        std = np.full(total.shape, np.nan)
    data = np.vstack([mean, std, np.asarray(moments.min, dtype=np.float64), np.asarray(moments.max, dtype=np.float64)])
    return pd.DataFrame(data, index=['mean', 'std', 'min', 'max'], columns=_labels(('Pan', 'Core'), num_strains),
                        copy=False)


def shared_gene_counts(df_genes, device=None):
    '''
    Genome x genome shared-gene matrix S = X^T X of a binary gene x genome table: S[k, l] is the number of genes
    present in both genome k and genome l, S[k, k] the genes of genome k.  The start of clustering genomes by gene
    content, Jaccard distances and genomic fluidity.  Computed on the GPU from the table's plan (shared with
    estimate_pan_core_size / estimate_pan_core_summary, so the table is not planned again), the dense part as an
    8-bit integer matrix product on the tensor cores.  Prints nothing and leaves ``np.random`` untouched.

    Returns
    -------
    df_shared : pd.DataFrame
        int32, N x N, index and columns ``df_genes.columns``.
    '''
    engine = _engine_for(df_genes, device)
    shared = engine.shared_genes_device().cpu().numpy()
    return pd.DataFrame(shared, index=df_genes.columns, columns=df_genes.columns, copy=False)


def compute_genomic_fluidity(df_genes, device=None):
    '''
    Genomic fluidity (Kislyuk, Haegeman, Bergman & Weitz, BMC Genomics 12:32, 2011): the mean over genome pairs of
    the share of their genes that the two genomes do not share, (|U_k| + |U_l|) / (M_k + M_l) with U the genes of one
    genome absent from the other and M the genomes' gene counts.  Unlike Heaps' alpha from rarefaction it does not
    depend on the order genomes were sampled in.  Its standard error is the leave-one-genome-out jackknife.

    The shared-gene matrix and the per-genome sums of the pair distances are computed on the GPU (see
    shared_gene_counts); only N numbers come back to the host.  Prints nothing and leaves ``np.random`` untouched.

    Returns
    -------
    pd.Series
        float64 entries ``fluidity``, ``jackknife_se`` (NaN for two genomes) and ``n_genomes``.  Tables of fewer
        than two genomes raise ValueError.
    '''
    _, num_strains = df_genes.shape
    if num_strains < 2:
        raise ValueError("genomic fluidity needs at least two genomes, got %d" % num_strains)
    engine = _engine_for(df_genes, device)
    rows = engine.fluidity_rows_device(engine.shared_genes_device()).cpu().numpy()
    return fluidity_series(rows)


def fluidity_series(row_sums):
    """The Series of compute_genomic_fluidity() from R[k] = sum over l != k of the pair distances d_kl:
    T = fsum(R) / 2 is the sum over pairs, fluidity = T / C(N, 2), leave-one-genome-out values
    (T - R[i]) / C(N - 1, 2) and jackknife_se = sqrt((N - 1) / N * sum((phi_i - mean phi)^2))."""
    rows = np.asarray(row_sums, dtype=np.float64)
    n = int(rows.shape[0])
    if n < 2:
        raise ValueError("genomic fluidity needs at least two genomes, got %d" % n)
    total = math.fsum(rows) / 2
    fluidity = total / (n * (n - 1) / 2)
    if n > 2:
        loo = (total - rows) / ((n - 1) * (n - 2) / 2)
        se = math.sqrt((n - 1) / n * float(np.sum((loo - loo.mean()) ** 2)))
    else:
        se = np.nan
    return pd.Series({'fluidity': fluidity, 'jackknife_se': se, 'n_genomes': float(n)}, dtype=np.float64)


def compute_bernoulli_grid_core_genome(df_genes_dense,
    prob_bounds=(0.8,0.99999999), init_capture_prob=0.9999,
    init_gene_freqs=None, device=None):
    '''
    Bernoulli-grid maximum likelihood: gene i has true frequency p_i, genome j captures
    genes at rate q_j, X_ij ~ Bernoulli(p_i q_j).  P and Q are fitted with L-BFGS-B.

    Parameters and returns are those of the reference (:101-166): a dense binary
    gene x genome DataFrame in, ``(df_opt, res)`` out, where df_opt has index
    ['Loglikelihood', 'p_<gene>'..., 'q_<genome>'...] and columns ['initial', 'optimum'],
    and res is scipy's OptimizeResult.
    '''
    n_genes, n_genomes = df_genes_dense.shape
    X = df_genes_dense.values
    grid = BernoulliGrid(X, device=device)
    if init_gene_freqs is None:
        P_guess = grid.row_count / float(n_genomes)
    else:
        P_guess = np.array(init_gene_freqs)
    Q_guess = init_capture_prob * np.ones(n_genomes)
    PQ_guess = np.clip(np.concatenate((P_guess, Q_guess)), prob_bounds[0], prob_bounds[1])
    init_ll = grid.ll_grad(PQ_guess)[0]
    print('Initial loglikelihood:', init_ll)

    labels = ['Loglikelihood'] + ['p_' + x for x in df_genes_dense.index] \
        + ['q_' + x for x in df_genes_dense.columns]
    df_init = pd.Series(data=[init_ll] + PQ_guess.tolist(), index=labels)
    df_init.name = 'initial'

    neg_ll = lambda PQ: -grid.ll_grad(PQ)[0]
    neg_ll_grad = lambda PQ: -grid.ll_grad(PQ)[1]
    bounds = [prob_bounds] * len(PQ_guess)
    res = scipy.optimize.minimize(neg_ll, PQ_guess, method='L-BFGS-B', jac=neg_ll_grad,
                                  bounds=bounds, options={'disp': True})
    print('Final loglikelihood:', -res.fun)
    df_opt = pd.Series(data=[-res.fun] + res.x.tolist(), index=labels)
    df_opt.name = 'optimum'
    return pd.concat([df_init, df_opt], axis=1), res


def __bernoulli_grid_loglikelihood__(X, P, Q):
    ''' LL of the observed table X for gene frequencies P and capture rates Q (GPU, fp64). '''
    return BernoulliGrid(X).loglikelihood(np.asarray(P, dtype=np.float64), np.asarray(Q, dtype=np.float64))


def __bernoulli_grid_loglikelihood_gradient__(X, P, Q):
    ''' Gradient of the LL with respect to concat(P, Q) (GPU, fp64). '''
    return BernoulliGrid(X).gradient(np.asarray(P, dtype=np.float64), np.asarray(Q, dtype=np.float64))


def compute_beta_binomial_core_genome(df_genes, frac_recovered=0.999, df_counts=None,
                                      num_points=100, ks_iter=1000, device=None):
    '''
    Frequency threshold for core genes from an error-rate model: the number of genomes a core gene is
    missing from is modelled as BetaBinomial(n_genomes, alpha, beta), fitted by maximum likelihood to the
    ``num_points`` highest gene frequencies.

    Parameters, return value (a Series for one ``num_points``, a DataFrame indexed by the number of points for a
    list; entries alpha, beta, cutoff, mae, kolmogorov_smirnov_pvalue, shapiro_wilk_pvalue, durbin_watson_stat)
    and the use of the global numpy RNG are those of the reference (:295-400).  ``df_genes`` may be the
    reference's binary DataFrame with SparseArray columns or a LightSparseDataFrame (anything with a scipy
    ``.data``); its gene-frequency spectrum is counted on the GPU and ordered by first appearance among the
    genes, like the collections.Counter of :355.  The Monte-Carlo KS simulation runs on the GPU.
    '''
    if df_counts is None:
        n_genes, n_genomes = df_genes.shape
        df_counts = _gene_frequency_spectrum(df_genes, device)
    else:
        n_genomes = max(df_counts.index)

    fitted = {}
    fit_points = num_points if type(num_points) != int else [num_points]      # noqa: E721 (bool / np.int64 as in :359)
    for n_points in fit_points:
        # :364-366 -- the last n_points entries of the spectrum AS ORDERED, frequencies -> misses, reversed
        tail = df_counts.iloc[-n_points:]
        misses = n_genomes - tail.index
        df = pd.Series(tail.values, index=misses).reindex(misses[::-1])
        X = np.asarray(df.index)
        Y = df.values

        neg_ll = lambda ab: -np.dot(Y, betabin_logpmf(X, n_genomes, ab[0], ab[1]))      # noqa: E731
        a, b = scipy.optimize.minimize(neg_ll, x0=(1, 100), method='Nelder-Mead').x

        cutoff = 0
        cdf = np.exp(betabin_logpmf(cutoff, n_genomes, a, b))
        while cdf < frac_recovered:
            cutoff += 1
            cdf += np.exp(betabin_logpmf(cutoff, n_genomes, a, b))

        residuals = np.asarray(Y - Y.sum() * np.exp(betabin_logpmf(X, n_genomes, a, b)))
        mae = np.abs(residuals).mean()
        sw_pvalue = scipy.stats.shapiro(residuals)[1]
        dwstat = _durbin_watson(residuals)

        model_cdf = np.cumsum(np.exp(betabin_logpmf(np.arange(n_genomes), n_genomes, a, b)))
        sim_limit = np.where(1 - model_cdf < 1e-8)[0][0]           # simulate up to tolerance 1e-8 (:386)
        if sim_limit > 0:
            ks_pvalue = ks_montecarlo_bbn(df, n_genomes, a, b, iterations=ks_iter, sim_limit=sim_limit,
                                          device=device)[0]
        else:
            ks_pvalue = np.nan
        fitted[n_points] = pd.Series({
            'alpha': a, 'beta': b, 'cutoff': cutoff, 'mae': mae,
            'kolmogorov_smirnov_pvalue': ks_pvalue,
            'shapiro_wilk_pvalue': sw_pvalue,
            'durbin_watson_stat': dwstat})
    table = pd.DataFrame.from_dict(fitted, orient='index')
    return table.iloc[0, :] if table.shape[0] == 1 else table


def _gene_frequency_spectrum(df_genes, device=None):
    """{gene frequency: number of genes} as the reference builds it at :352-355 -- a collections.Counter over
    the row sums, i.e. keyed in order of FIRST APPEARANCE among the genes -- from GPU counts."""
    from . import sparse_utils
    from .engine import table_marginals
    data = df_genes.data if hasattr(df_genes, 'data') and hasattr(df_genes.data, 'tocoo') \
        else sparse_utils.sparse_arrays_to_spmatrix(df_genes)
    _, _, spectrum, first_gene = table_marginals(data, device=device)
    present = np.flatnonzero(spectrum)
    order = present[np.argsort(first_gene[present], kind='stable')]
    return pd.Series(collections.OrderedDict((int(m), int(spectrum[m])) for m in order), dtype=np.int64)


def _durbin_watson(residuals):
    """statsmodels.stats.stattools.durbin_watson (:380) where statsmodels is installed, else its definition."""
    try:
        from statsmodels.stats.stattools import durbin_watson
    except ImportError:
        residuals = np.asarray(residuals, dtype=np.float64)
        return float(np.sum(np.diff(residuals) ** 2) / np.sum(residuals ** 2))
    return durbin_watson(residuals)


def ks_montecarlo_bbn(Ycounts, n, a, b, iterations=100, sim_limit=1000, device=None):
    '''
    Monte-Carlo Kolmogorov-Smirnov test for a beta-binomial (:457-482): the KS statistic of the observed
    counts against BBN(n, a, b) and its distribution under the model, simulated with ``iterations`` samples of
    ``Ycounts.sum()`` draws each.  Returns (pvalue, ks_stat, ks_sim).  The draws come from the global numpy RNG
    exactly as the reference's ``np.random.choice`` takes them; drawing, eCDFs and statistics run on the GPU.
    '''
    from .engine import ks_montecarlo_statistics
    support = np.arange(sim_limit)
    model_cdf = np.cumsum(np.exp(betabin_logpmf(support, n, a, b)))
    ks_stat = np.max(np.abs(ecdf_from_counts(Ycounts.index, Ycounts.values, sim_limit) - model_cdf))

    n_samples = Ycounts.sum()
    iterations = int(iterations)
    probs = _bbn_probabilities(n, a, b, sim_limit)
    if n_samples * iterations <= 0:
        ks_sim = np.full(max(iterations, 0), np.nan)               # the reference divides an empty eCDF by zero
    else:
        choice_cdf = probs.cumsum()                                # numpy legacy RandomState.choice
        choice_cdf /= choice_cdf[-1]
        ks_sim = ks_montecarlo_statistics(choice_cdf, model_cdf, n_samples, iterations, device=device)
    pvalue = (ks_stat < ks_sim).sum() / float(iterations)
    return pvalue, ks_stat, ks_sim


def _bbn_probabilities(n, a, b, sim_limit):
    """The probabilities draw_bbn hands to np.random.choice (:489-491), with numpy's own argument checks."""
    probs = np.exp(betabin_logpmf(np.arange(sim_limit), n, a, b))
    probs /= probs.sum()
    if np.isnan(probs).any():
        raise ValueError("probabilities contain NaN")
    if (probs < 0).any():
        raise ValueError("probabilities are not non-negative")
    return probs


def draw_bbn(n, a, b, size, sim_limit=1000):
    '''
    ``size`` draws from BBN(n, a, b) truncated to 0 .. sim_limit - 1 (:484-492), from the global numpy RNG.
    '''
    return np.random.choice(np.arange(sim_limit), size=size, p=_bbn_probabilities(n, a, b, sim_limit))


def ecdf_from_counts(vals, counts, limit):
    ''' eCDF on 0 .. limit - 1 from unique values and their counts (:494-499). '''
    pmf = np.zeros(limit)
    vals = np.asarray(vals)
    if vals.size and (vals.max() >= limit or vals.min() < -limit):
        raise IndexError('index %d is out of bounds for axis 0 with size %d' % (int(vals.max()), limit))
    np.add.at(pmf, vals, counts)
    return np.cumsum(pmf) / pmf.sum()


def betabin_logpmf(x, n, a, b):
    ''' Beta-binomial log-PMF (:501-508; scipy.stats.betabinom._logpmf). '''
    k = np.floor(x)
    return -np.log(n + 1) - betaln(n - k + 1, k + 1) + betaln(k + a, n - k + b) - betaln(a, b)
