"""ctypes binding of libpeaksegdisk_b200.so (the C ABI in include/peaksegdisk_b200.h).

The library is built in-tree by `__graft_entry__.build()` / `make -C peaksegdisk_b200/csrc`.  There is
no Python or CPU fallback: if the shared object is missing, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PSD_LIB") or os.path.join(_HERE, "libpeaksegdisk_b200.so")   # PSD_LIB: kernel-variant experiments


class PsdResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("trivial", C.c_int32), ("n_rows", C.c_int32), ("n_segments", C.c_int32),
                ("n_peaks", C.c_int32), ("n_equality", C.c_int32), ("penalty", C.c_double), ("bases", C.c_double),
                ("mean_pen_cost", C.c_double), ("total_loss", C.c_double), ("mean_intervals", C.c_double),
                ("max_intervals", C.c_double)]


class PsdStats(C.Structure):
    _fields_ = [("dp_ms", C.c_double), ("backtrack_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
                ("rows_solved", C.c_int64), ("store_bytes_algorithmic", C.c_int64), ("store_bytes_written", C.c_int64),
                ("store_bytes_spilled_host", C.c_int64),
                ("backtrack_bytes_read", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("n_launches", C.c_int32), ("n_waves", C.c_int32), ("n_overflow_tier", C.c_int32),
                ("piece_cap", C.c_int32), ("warps_per_sm", C.c_int32), ("n_sm", C.c_int32),
                ("n_rle_launches", C.c_int32), ("rle_ms", C.c_double), ("rle_positions", C.c_int64),
                ("rle_bytes_algorithmic", C.c_int64), ("n_latency_waves", C.c_int32), ("pad_", C.c_int32),
                ("store_bytes_drained_dma", C.c_int64)]


class PsdBatchStats(C.Structure):
    _fields_ = [("parse_ms", C.c_double), ("build_ms", C.c_double), ("run_ms", C.c_double), ("write_ms", C.c_double),
                ("release_ms", C.c_double), ("dp_ms", C.c_double), ("backtrack_ms", C.c_double),
                ("rows_parsed", C.c_int64), ("rows_solved", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("store_bytes_algorithmic", C.c_int64), ("n_problems", C.c_int32), ("n_files_parsed", C.c_int32),
                ("n_devices", C.c_int32), ("n_launches", C.c_int32), ("n_waves", C.c_int32), ("n_latency_waves", C.c_int32)]


class PsdReads(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("read_start", C.POINTER(C.c_int32)), ("read_end", C.POINTER(C.c_int32)),
                ("region_start", C.c_int32), ("region_end", C.c_int32)]


class PsdCoverageStats(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("kernel_ms", C.c_double), ("reads", C.c_int64), ("bases", C.c_int64),
                ("rows", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("n_problems", C.c_int32),
                ("n_waves", C.c_int32)]


class PsdLabelErrors(C.Structure):
    _fields_ = [("fp", C.c_int32), ("fn", C.c_int32), ("possible_fp", C.c_int32), ("possible_fn", C.c_int32),
                ("errors", C.c_int32)]


class PsdPathProblem(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("chromStart", C.POINTER(C.c_int32)), ("chromEnd", C.POINTER(C.c_int32)),
                ("coverage", C.POINTER(C.c_int32)), ("n_labels", C.c_int64), ("label_start", C.POINTER(C.c_int32)),
                ("label_end", C.POINTER(C.c_int32)), ("label_kind", C.POINTER(C.c_int32))]


class PsdPathModel(C.Structure):
    _fields_ = [("min_lambda", C.c_double), ("max_lambda", C.c_double), ("penalty", C.c_double), ("total_loss", C.c_double),
                ("peaks", C.c_int32), ("segments", C.c_int32), ("fp", C.c_int32), ("fn", C.c_int32),
                ("possible_fp", C.c_int32), ("possible_fn", C.c_int32), ("errors", C.c_int32), ("pad_", C.c_int32)]


class PsdPathStats(C.Structure):
    _fields_ = [("dp_ms", C.c_double), ("backtrack_ms", C.c_double), ("label_ms", C.c_double), ("rows_solved", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("rounds", C.c_int32), ("solves", C.c_int32),
                ("models", C.c_int32), ("n_problems", C.c_int32)]


class PsdRows(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("chromStart", C.POINTER(C.c_int32)), ("chromEnd", C.POINTER(C.c_int32)),
                ("coverage", C.POINTER(C.c_int32))]


class PsdProblemFeatures(C.Structure):
    _fields_ = [("quartile", C.c_double * 5), ("mean", C.c_double), ("sd", C.c_double), ("bases", C.c_int64),
                ("rows", C.c_int64)]


class PsdFeaturesStats(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("kernel_ms", C.c_double), ("rows", C.c_int64), ("h2d_bytes", C.c_int64),
                ("d2h_bytes", C.c_int64), ("n_problems", C.c_int32), ("n_waves", C.c_int32), ("n_launches", C.c_int32)]


class PsdJointSample(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("chromStart", C.POINTER(C.c_int32)), ("chromEnd", C.POINTER(C.c_int32)),
                ("coverage", C.POINTER(C.c_int32)), ("n_labels", C.c_int64), ("label_start", C.POINTER(C.c_int32)),
                ("label_end", C.POINTER(C.c_int32)), ("label_kind", C.POINTER(C.c_int32))]


class PsdJointProblem(C.Structure):
    _fields_ = [("region_start", C.c_int32), ("region_end", C.c_int32), ("bin_bases", C.c_int32), ("n_samples", C.c_int32),
                ("samples", C.POINTER(PsdJointSample))]


class PsdJointModel(C.Structure):
    _fields_ = [("total_loss", C.c_double), ("min_lambda", C.c_double), ("max_lambda", C.c_double), ("peaks", C.c_int32),
                ("peak_start", C.c_int32), ("peak_end", C.c_int32), ("selectable", C.c_int32), ("fp", C.c_int32),
                ("fn", C.c_int32), ("possible_fp", C.c_int32), ("possible_fn", C.c_int32), ("errors", C.c_int32),
                ("pad_", C.c_int32)]


class PsdJointStats(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("kernel_ms", C.c_double), ("samples", C.c_int64), ("pair_sample_evals", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("n_problems", C.c_int32), ("n_waves", C.c_int32),
                ("n_launches", C.c_int32), ("pad_", C.c_int32)]


# every symbol include/peaksegdisk_b200.h declares (tests check the library exports all of them)
C_ABI_SYMBOLS = [
    "psd_fpop_disk", "psd_fpop_disk_batch", "psd_status_message", "psd_last_error", "psd_plan_create",
    "psd_plan_destroy", "psd_plan_add", "psd_plan_add_counts", "psd_plan_size", "psd_plan_upload", "psd_plan_solve", "psd_plan_download",
    "psd_plan_run", "psd_plan_result", "psd_plan_segments", "psd_plan_get_stats", "psd_plan_set_penalty", "psd_plan_store_function", "psd_write_bedgraph", "psd_last_batch_stats",
    "psd_set_option", "psd_device_count", "psd_release_cache",
    "psd_coverage_from_reads", "psd_coverage_n_rows", "psd_coverage_rows", "psd_coverage_get_stats", "psd_coverage_free",
    "psd_plan_set_labels", "psd_plan_label_errors", "psd_model_path", "psd_path_status", "psd_path_n_models",
    "psd_path_models", "psd_path_target", "psd_path_get_stats", "psd_path_free", "psd_features",
    "psd_joint_models", "psd_joint_n_models", "psd_joint_model_table", "psd_joint_samples", "psd_joint_target",
    "psd_joint_get_stats", "psd_joint_free",
    "_Z16PeakSegFPOP_diskPcS_S_",   # the reference's own C++-linkage entry (src/PeakSegFPOPLog.h:15)
]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "peaksegdisk_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    i32p, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    lib.psd_fpop_disk.restype = C.c_int
    lib.psd_fpop_disk.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
    lib.psd_fpop_disk_batch.restype = C.c_int
    lib.psd_fpop_disk_batch.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                        C.POINTER(C.c_int)]
    lib.psd_status_message.restype = C.c_char_p
    lib.psd_status_message.argtypes = [C.c_int]
    lib.psd_last_error.restype = C.c_char_p
    lib.psd_plan_create.restype = C.c_void_p
    lib.psd_plan_create.argtypes = [C.c_int]
    lib.psd_plan_destroy.restype = None
    lib.psd_plan_destroy.argtypes = [C.c_void_p]
    lib.psd_plan_add.restype = C.c_int
    lib.psd_plan_add.argtypes = [C.c_void_p, C.c_int64, i32p, i32p, i32p, C.c_double, C.c_int]
    lib.psd_plan_add_counts.restype = C.c_int
    lib.psd_plan_add_counts.argtypes = [C.c_void_p, C.c_int64, i32p, C.c_double, C.c_int]
    lib.psd_release_cache.restype = None
    lib.psd_release_cache.argtypes = []
    lib.psd_plan_size.restype = C.c_int
    lib.psd_plan_size.argtypes = [C.c_void_p]
    for name in ("psd_plan_upload", "psd_plan_solve", "psd_plan_download", "psd_plan_run"):
        f = getattr(lib, name)
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_void_p]
    lib.psd_plan_result.restype = C.c_int
    lib.psd_plan_result.argtypes = [C.c_void_p, C.c_int, C.POINTER(PsdResult)]
    lib.psd_plan_segments.restype = C.c_int
    lib.psd_plan_segments.argtypes = [C.c_void_p, C.c_int, i32p, i32p, i32p, dp]
    lib.psd_plan_get_stats.restype = C.c_int
    lib.psd_plan_get_stats.argtypes = [C.c_void_p, C.POINTER(PsdStats)]
    lib.psd_plan_set_penalty.restype = C.c_int
    lib.psd_plan_set_penalty.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_int]
    lib.psd_plan_store_function.restype = C.c_int
    lib.psd_plan_store_function.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, i32p, dp, i32p, dp]
    lib.psd_last_batch_stats.restype = C.c_int
    lib.psd_last_batch_stats.argtypes = [C.POINTER(PsdBatchStats)]
    lib.psd_write_bedgraph.restype = C.c_int
    lib.psd_write_bedgraph.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, i32p, i32p, i32p]
    lib.psd_set_option.restype = C.c_int
    lib.psd_set_option.argtypes = [C.c_char_p, C.c_double]
    lib.psd_device_count.restype = C.c_int
    lib.psd_coverage_from_reads.restype = C.c_int
    lib.psd_coverage_from_reads.argtypes = [C.c_int, C.c_int, C.POINTER(PsdReads), C.POINTER(C.c_void_p)]
    lib.psd_coverage_n_rows.restype = C.c_int64
    lib.psd_coverage_n_rows.argtypes = [C.c_void_p, C.c_int]
    lib.psd_coverage_rows.restype = C.c_int
    lib.psd_coverage_rows.argtypes = [C.c_void_p, C.c_int, i32p, i32p, i32p]
    lib.psd_coverage_get_stats.restype = C.c_int
    lib.psd_coverage_get_stats.argtypes = [C.c_void_p, C.POINTER(PsdCoverageStats)]
    lib.psd_coverage_free.restype = None
    lib.psd_coverage_free.argtypes = [C.c_void_p]
    lib.psd_plan_set_labels.restype = C.c_int
    lib.psd_plan_set_labels.argtypes = [C.c_void_p, C.c_int, C.c_int64, i32p, i32p, i32p]
    lib.psd_plan_label_errors.restype = C.c_int
    lib.psd_plan_label_errors.argtypes = [C.c_void_p, C.c_int, C.POINTER(PsdLabelErrors), i32p, i32p]
    lib.psd_model_path.restype = C.c_int
    lib.psd_model_path.argtypes = [C.c_int, C.c_int, C.POINTER(PsdPathProblem), C.c_double, C.c_double, C.POINTER(C.c_void_p)]
    lib.psd_path_status.restype = C.c_int
    lib.psd_path_status.argtypes = [C.c_void_p, C.c_int]
    lib.psd_path_n_models.restype = C.c_int
    lib.psd_path_n_models.argtypes = [C.c_void_p, C.c_int]
    lib.psd_path_models.restype = C.c_int
    lib.psd_path_models.argtypes = [C.c_void_p, C.c_int, C.POINTER(PsdPathModel)]
    lib.psd_path_target.restype = C.c_int
    lib.psd_path_target.argtypes = [C.c_void_p, C.c_int, dp, dp, i32p]
    lib.psd_path_get_stats.restype = C.c_int
    lib.psd_path_get_stats.argtypes = [C.c_void_p, C.POINTER(PsdPathStats)]
    lib.psd_path_free.restype = None
    lib.psd_path_free.argtypes = [C.c_void_p]
    lib.psd_features.restype = C.c_int
    lib.psd_features.argtypes = [C.c_int, C.c_int, C.POINTER(PsdRows), C.POINTER(PsdProblemFeatures),
                                 C.POINTER(PsdFeaturesStats)]
    lib.psd_joint_models.restype = C.c_int
    lib.psd_joint_models.argtypes = [C.c_int, C.c_int, C.POINTER(PsdJointProblem), C.POINTER(C.c_void_p)]
    lib.psd_joint_n_models.restype = C.c_int
    lib.psd_joint_n_models.argtypes = [C.c_void_p, C.c_int]
    lib.psd_joint_model_table.restype = C.c_int
    lib.psd_joint_model_table.argtypes = [C.c_void_p, C.c_int, C.POINTER(PsdJointModel)]
    lib.psd_joint_samples.restype = C.c_int
    lib.psd_joint_samples.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_uint8)]
    lib.psd_joint_target.restype = C.c_int
    lib.psd_joint_target.argtypes = [C.c_void_p, C.c_int, dp, dp, i32p]
    lib.psd_joint_get_stats.restype = C.c_int
    lib.psd_joint_get_stats.argtypes = [C.c_void_p, C.POINTER(PsdJointStats)]
    lib.psd_joint_free.restype = None
    lib.psd_joint_free.argtypes = [C.c_void_p]
    return lib


lib = _load()


def status_text(status, bedgraph="", penalty="", db=""):
    """The error text src/interface.cpp:16-55 raises for a status code."""
    fmt = lib.psd_status_message(status).decode()
    if status in (1, 2, 10):
        return fmt % penalty
    if status in (3, 4, 5, 6, 9):
        return fmt % bedgraph
    if status == 7:
        return fmt % db
    if status in (8, 11):
        return fmt % (bedgraph, penalty)
    if "%d" in fmt:
        return fmt % status
    extra = lib.psd_last_error().decode()
    return fmt + (": " + extra if extra else "")


def last_batch_stats():
    """Stage times and device counters of the process's last file-batch call, as a dict."""
    st = PsdBatchStats()
    lib.psd_last_batch_stats(C.byref(st))
    return {name: getattr(st, name) for name, _ in st._fields_}
