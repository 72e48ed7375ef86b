"""abo_b200 — B200-native GP-surrogate + acquisition hot path behind the AbstractBayesOpt.jl
plug-in API (AbstractSurrogate / AbstractAcquisition / AbstractDomain).  The compute lives in
the hand-written sm_100a library `libabo_cuda.so` (csrc/, C ABI in include/abo.h); this package
is the host-side mirror of the reference interface for that path.  No CPU fallback."""
from ._lib import (AboCudaError, Context, DimensionMismatch, GpHandle, PosDefException, default_context,
                   nccl_unique_id, LIB_PATH, SYMBOLS)
from .kernels import (ADMatern52Kernel, ADMatern72Kernel, ApproxMatern52Kernel, ApproxMatern72Kernel, Kernel,
                      Matern52Kernel, Matern72Kernel, SqExponentialKernel, with_lengthscale,
                      extract_scale_and_lengthscale)
from .surrogates import (AbstractSurrogate, GradientGP, StandardGP, get_kernel_constructor, get_lengthscale,
                         get_mean_std, get_scale, is_ard, nlml, nlml_batch, nlml_ls, posterior_grad_mean,
                         posterior_grad_var, posterior_grad_cov, posterior_cov, posterior_mean, posterior_sample, posterior_var,
                         max_value_samples, pathwise_sample, pathwise_thompson_batch, prep_input, prep_output, rescale_model,
                         std_y, thompson_batch, unstandardized_mean_and_var, update_surrogate, empty_posterior_like, _get_minimum,
                         _update_model_parameters)
from .acquisition import (AbstractAcquisition, EnsembleAcquisition, ExpectedImprovement, GradientNormUCB,
                          MaxValueEntropySearch, PathwiseThompsonSampling, ProbabilityImprovement, ThompsonSampling,
                          UpperConfidenceBound, qExpectedImprovement)
from .domains import AbstractDomain, ContinuousDomain
from .parallel import (init_nccl_context, merge_topk, shard_range, sharded_nlml_batch, sharded_restarts, sharded_topk,
                       sync_posterior)
from .bayesian_opt import (BOStruct, latin_hypercube, lengthscale_bounds, lockstep_lbfgsb, monte_carlo_fill_distance, optimize, optimize_acquisition, optimize_hyperparameters,
                           print_info, rescale_output, standardize_problem, stop_criteria, update_bo)


def update(obj, *args, **kw):
    """`update` as the reference overloads it by dispatch: update(model, xs, ys) → new model;
    update(acq, ys, model) → new acquisition; update(BO, x, y, i) → BO."""
    if isinstance(obj, AbstractSurrogate):
        return update_surrogate(obj, *args, **kw)
    if isinstance(obj, AbstractAcquisition):
        return obj.update(*args)
    if isinstance(obj, BOStruct):
        return update_bo(obj, *args)
    raise TypeError(f"no method update({type(obj).__name__}, ...)")


def copy(obj):
    return obj.copy()
