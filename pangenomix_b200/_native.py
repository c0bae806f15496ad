"""ctypes binding of libpgx_b200.so (the C ABI declared in include/pgx.h).

There is no fallback: if the shared object is missing or a call fails, the caller gets an
exception, never a CPU result.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PGX_LIBRARY selects another build of the SAME library (scripts/sanitize_host.sh: host helpers under ASan/UBSan)
LIB_PATH = os.environ.get("PGX_LIBRARY") or os.path.join(_HERE, "libpgx_b200.so")

# every symbol include/pgx.h declares (tests check the library exports all of them)
EXPORTS = (
    "pgx_version", "pgx_last_error", "pgx_device_info", "pgx_pan_core_curves",
    "pgx_pan_core_curves_f64", "pgx_pan_core_curves_host", "pgx_set_tuning",
    "pgx_launch_count", "pgx_bernoulli_scratch_bytes", "pgx_bernoulli_ll_grad",
    "pgx_legacy_shuffles", "pgx_profile_enable", "pgx_profile_read",
    "pgx_heaps_scratch_bytes", "pgx_heaps_fit", "pgx_estimate_pan_core",
    "pgx_plan_all_equal_u64", "pgx_inflate_raw",
    "pgx_expand_deltas", "pgx_host_plan_create", "pgx_host_plan_destroy", "pgx_plan_create", "pgx_plan_upload",
    "pgx_plan_destroy", "pgx_set_trace", "pgx_legacy_random_raw", "pgx_coo_marginals", "pgx_frequency_spectrum",
    "pgx_coo_marginals_host", "pgx_ks_scratch_bytes", "pgx_ks_montecarlo", "pgx_ks_montecarlo_host", "pgx_expand_split", "pgx_split_head",
    "pgx_random_perms", "pgx_curve_moments", "pgx_shared_genes", "pgx_fluidity_rows",
    "pgx_plan_spectrum", "pgx_pair_overlap_histograms", "pgx_pair_overlap_work_bytes", "pgx_rarefaction_moments",
)


class PgxError(RuntimeError):
    """A libpgx_b200 call returned a non-zero status."""


class PgxPlan(ctypes.Structure):
    """Mirror of ``struct pgx_plan`` (include/pgx.h)."""
    _fields_ = [
        ("d_chunks", ctypes.c_void_p),
        ("d_tasks", ctypes.c_void_p),
        ("d_sorted_idx", ctypes.c_void_p),
        ("d_sorted_ptr", ctypes.c_void_p),
        ("d_bits", ctypes.c_void_p),
        ("reserved_ptr", ctypes.c_void_p),
        ("d_colsum", ctypes.c_void_p),
        ("d_w_present", ctypes.c_void_p),
        ("d_w_absent", ctypes.c_void_p),
        ("n_chunks", ctypes.c_int64),
        ("n_genomes", ctypes.c_int32),
        ("n_genes", ctypes.c_int32),
        ("n_rows", ctypes.c_int32),
        ("n_tasks", ctypes.c_int32),
        ("n_long", ctypes.c_int32),
        ("n_superblocks", ctypes.c_int32),
        ("perms_per_cta", ctypes.c_int32),
        ("slice_words", ctypes.c_int32),
        ("max_colsum", ctypes.c_int32),
        ("reserved_i32", ctypes.c_int32),
    ]


class PgxHostPlan(ctypes.Structure):
    """Mirror of ``struct pgx_host_plan`` (include/pgx.h)."""
    _fields_ = [
        ("owner", ctypes.c_void_p),
        ("chunks", ctypes.c_void_p),
        ("tasks", ctypes.c_void_p),
        ("sorted_idx", ctypes.c_void_p),
        ("sorted_ptr", ctypes.c_void_p),
        ("bits", ctypes.c_void_p),
        ("colsum", ctypes.c_void_p),
        ("w_present", ctypes.c_void_p),
        ("w_absent", ctypes.c_void_p),
        ("row_gene", ctypes.c_void_p),
        ("row_len", ctypes.c_void_p),
        ("row_absent", ctypes.c_void_p),
        ("long_gene", ctypes.c_void_p),
        ("nnz", ctypes.c_int64),
        ("nnz_list", ctypes.c_int64),
        ("nnz_long", ctypes.c_int64),
        ("n_chunks", ctypes.c_int64),
        ("n_bits_words", ctypes.c_int64),
        ("n_sorted", ctypes.c_int64),
        ("n_genomes", ctypes.c_int32),
        ("n_genes", ctypes.c_int32),
        ("n_rows", ctypes.c_int32),
        ("n_tasks", ctypes.c_int32),
        ("n_long", ctypes.c_int32),
        ("n_superblocks", ctypes.c_int32),
        ("perms_per_cta", ctypes.c_int32),
        ("slice_words", ctypes.c_int32),
        ("long_threshold", ctypes.c_int32),
        ("max_colsum", ctypes.c_int32),
        ("n_empty", ctypes.c_int32),
        ("n_full", ctypes.c_int32),
    ]


_lib = None


def load():
    """Loads the library once; raises if it has not been built (python -m pangenomix_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PgxError(
            "%s is missing: build it with `python -m pangenomix_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    plan_p = ctypes.POINTER(PgxPlan)
    lib.pgx_version.restype = ctypes.c_int
    lib.pgx_version.argtypes = []
    lib.pgx_last_error.restype = ctypes.c_char_p
    lib.pgx_last_error.argtypes = []
    lib.pgx_device_info.restype = ctypes.c_int
    lib.pgx_device_info.argtypes = [ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i64)]
    lib.pgx_pan_core_curves.restype = ctypes.c_int
    lib.pgx_pan_core_curves.argtypes = [plan_p, vp, i64, vp, vp]
    lib.pgx_pan_core_curves_f64.restype = ctypes.c_int
    lib.pgx_pan_core_curves_f64.argtypes = [plan_p, vp, i64, vp, vp, vp]
    lib.pgx_pan_core_curves_host.restype = ctypes.c_int
    lib.pgx_pan_core_curves_host.argtypes = [plan_p, vp, i64, vp, i32, i64]
    lib.pgx_set_trace.restype = ctypes.c_int
    lib.pgx_set_trace.argtypes = [vp, i64]
    lib.pgx_set_tuning.restype = ctypes.c_int
    lib.pgx_set_tuning.argtypes = [i32, i32, i32]
    lib.pgx_launch_count.restype = i64
    lib.pgx_launch_count.argtypes = []
    lib.pgx_bernoulli_scratch_bytes.restype = ctypes.c_size_t
    lib.pgx_bernoulli_scratch_bytes.argtypes = [i64, i64]
    lib.pgx_bernoulli_ll_grad.restype = ctypes.c_int
    lib.pgx_bernoulli_ll_grad.argtypes = [vp, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.pgx_plan_all_equal_u64.restype = ctypes.c_int
    lib.pgx_plan_all_equal_u64.argtypes = [vp, i64, ctypes.c_uint64, i32]
    lib.pgx_inflate_raw.restype = ctypes.c_int
    lib.pgx_inflate_raw.argtypes = [vp, i64, vp, i64]
    host_pp = ctypes.POINTER(ctypes.POINTER(PgxHostPlan))
    lib.pgx_host_plan_create.restype = ctypes.c_int
    lib.pgx_host_plan_create.argtypes = [vp, vp, i64, i32, i32, i32, i32, i32, host_pp]
    lib.pgx_host_plan_destroy.restype = None
    lib.pgx_host_plan_destroy.argtypes = [ctypes.POINTER(PgxHostPlan)]
    lib.pgx_plan_create.restype = ctypes.c_int
    lib.pgx_plan_create.argtypes = [vp, vp, i64, i32, i32, i32, ctypes.POINTER(plan_p)]
    lib.pgx_plan_upload.restype = ctypes.c_int
    lib.pgx_plan_upload.argtypes = [ctypes.POINTER(PgxHostPlan), ctypes.POINTER(plan_p)]
    lib.pgx_plan_destroy.restype = ctypes.c_int
    lib.pgx_plan_destroy.argtypes = [plan_p]
    lib.pgx_expand_deltas.restype = ctypes.c_int
    lib.pgx_expand_deltas.argtypes = [vp, i64, i32, vp, i32, i32]
    lib.pgx_split_head.restype = ctypes.c_int
    lib.pgx_split_head.argtypes = []
    lib.pgx_expand_split.restype = ctypes.c_int
    lib.pgx_expand_split.argtypes = [vp, i64, i32, i32, vp, i32, i32]
    lib.pgx_estimate_pan_core.restype = ctypes.c_int
    lib.pgx_estimate_pan_core.argtypes = [plan_p, vp, ctypes.POINTER(i32), i64, vp, i64]
    lib.pgx_heaps_scratch_bytes.restype = ctypes.c_size_t
    lib.pgx_heaps_scratch_bytes.argtypes = [i64]
    lib.pgx_heaps_fit.restype = ctypes.c_int
    lib.pgx_heaps_fit.argtypes = [vp, i32, i64, i64, i64, vp, vp, vp, vp]
    lib.pgx_legacy_shuffles.restype = ctypes.c_int
    lib.pgx_legacy_shuffles.argtypes = [vp, ctypes.POINTER(i32), i64, i64, vp]
    lib.pgx_legacy_random_raw.restype = ctypes.c_int
    lib.pgx_legacy_random_raw.argtypes = [vp, ctypes.POINTER(i32), i64, vp]
    lib.pgx_coo_marginals.restype = ctypes.c_int
    lib.pgx_coo_marginals.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp, i32, vp]
    lib.pgx_frequency_spectrum.restype = ctypes.c_int
    lib.pgx_frequency_spectrum.argtypes = [vp, i64, i32, vp, vp, vp]
    lib.pgx_coo_marginals_host.restype = ctypes.c_int
    lib.pgx_coo_marginals_host.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp, vp]
    lib.pgx_ks_scratch_bytes.restype = ctypes.c_size_t
    lib.pgx_ks_scratch_bytes.argtypes = [i64, i32]
    lib.pgx_ks_montecarlo.restype = ctypes.c_int
    lib.pgx_ks_montecarlo.argtypes = [vp, i64, i64, vp, vp, i32, vp, vp, vp]
    lib.pgx_ks_montecarlo_host.restype = ctypes.c_int
    lib.pgx_ks_montecarlo_host.argtypes = [vp, ctypes.POINTER(i32), i64, i64, vp, vp, i32, vp]
    lib.pgx_random_perms.restype = ctypes.c_int
    lib.pgx_random_perms.argtypes = [ctypes.c_uint64, i64, i64, i32, vp, vp]
    lib.pgx_curve_moments.restype = ctypes.c_int
    lib.pgx_curve_moments.argtypes = [vp, i64, i64, vp, vp, vp, vp, i32, vp]
    lib.pgx_shared_genes.restype = ctypes.c_int
    lib.pgx_shared_genes.argtypes = [plan_p, vp, vp, i64, vp]
    lib.pgx_fluidity_rows.restype = ctypes.c_int
    lib.pgx_fluidity_rows.argtypes = [vp, i32, vp, vp]
    lib.pgx_plan_spectrum.restype = ctypes.c_int
    lib.pgx_plan_spectrum.argtypes = [plan_p, vp, vp]
    lib.pgx_pair_overlap_histograms.restype = ctypes.c_int
    lib.pgx_pair_overlap_histograms.argtypes = [plan_p, vp, vp, vp, i64, vp]
    lib.pgx_pair_overlap_work_bytes.restype = i64
    lib.pgx_pair_overlap_work_bytes.argtypes = [i32, i64, i32]
    lib.pgx_rarefaction_moments.restype = ctypes.c_int
    lib.pgx_rarefaction_moments.argtypes = [vp, vp, vp, i64, i32, vp, vp]
    lib.pgx_profile_enable.restype = ctypes.c_int
    lib.pgx_profile_enable.argtypes = [i32]
    lib.pgx_profile_read.restype = ctypes.c_int
    lib.pgx_profile_read.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                     ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i64)]
    _lib = lib
    return lib


def check(status):
    if status != 0:
        message = load().pgx_last_error().decode("utf-8", "replace")
        raise PgxError("libpgx_b200 error %d: %s" % (status, message))


def launch_count():
    return int(load().pgx_launch_count())


def profile_enable(on=True):
    check(load().pgx_profile_enable(1 if on else 0))


def profile_read():
    """(list-kernel ms, probe-kernel ms, scan-kernel ms, calls) accumulated since the last read."""
    a, b, c, d = ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
    check(load().pgx_profile_read(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c), ctypes.byref(d)))
    return a.value, b.value, c.value, d.value


def set_tuning(perms_per_cta=0, row_splits=0, threads_per_cta=0):
    check(load().pgx_set_tuning(int(perms_per_cta), int(row_splits), int(threads_per_cta)))


def device_info():
    sm, smem, l2 = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int64()
    check(load().pgx_device_info(ctypes.byref(sm), ctypes.byref(smem), ctypes.byref(l2)))
    return {"sm_count": sm.value, "smem_optin_bytes": smem.value, "l2_bytes": l2.value}
