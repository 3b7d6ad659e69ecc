"""ggp-b200: B200-native (sm_100a, FP64) likelihood / forward-backward / joints recursion over cell
lineage trees, a drop-in for the hot path of bjks/gfp_gaussian_process.

Host-side mirror of the reference's entry points (same names and argument meaning):
  total_likelihood      likelihood.h:125-174
  prediction_forward / prediction_backward / combine_predictions   predictions.h:166, 438, 466
  collect_joint_distributions   correlation_tree.h:629
All numerical work is done by libggp_b200.so (hand-written CUDA); there is no CPU fallback.
"""
from .forest import Forest, ForestGroup, LineageData, NOISE_MODELS, DIVISION_MODELS, PARAM_NAMES  # noqa: F401
from .api import (total_likelihood, prediction_forward_backward, run_bound_1dscan, arange,  # noqa: F401
                  num_hessian_ll, total_likelihood_grad, total_likelihood_hess, num_hessian_grad, LikelihoodNaN, collect_joint_distributions, prediction_upper14, count_joints,
                  simulate_series, tree_scores, sandwich, sandwich_error_bars)
from .synthetic import simulate_forest, PARAMS_CONST_GAUSS, PARAMS_SCALED_BINOMIAL  # noqa: F401
from . import sharding  # noqa: F401
