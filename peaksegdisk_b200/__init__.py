"""peaksegdisk_b200 -- B200-native (sm_100a) PeakSegFPOP: one warp per (bedGraph x penalty) problem.

Public surface mirrors the reference R package for this path (api.py) plus the batched in-memory
Plan (plan.py).  All solves run in libpeaksegdisk_b200.so; importing fails if it is not built.
"""
from . import _lib
from .api import (PeakSegFPOP_file, PeakSegFPOP_file_batch, PeakSegFPOP_dir, PeakSegFPOP_df, PeakSegFPOP_vec,
                  PeakSegFPOP_vec_batch, coverage_from_reads,
                  sequentialSearch_dir, sequentialSearch_batch, writeBedGraph, col_name_list, r_paste)
from .plan import (Plan, solve_batch, solve_counts_batch, solve_reads_batch, model_path_batch, problem_features,
                   joint_models_batch)
from .learn import IntervalRegressionCV

__all__ = ["PeakSegFPOP_file", "PeakSegFPOP_file_batch", "PeakSegFPOP_dir", "PeakSegFPOP_df", "PeakSegFPOP_vec", "PeakSegFPOP_vec_batch",
           "sequentialSearch_dir", "sequentialSearch_batch", "writeBedGraph", "col_name_list", "r_paste", "Plan", "solve_batch",
           "solve_counts_batch", "coverage_from_reads", "solve_reads_batch", "model_path_batch",
           "problem_features", "joint_models_batch", "IntervalRegressionCV"]
