"""hmc.jl_b200 — B200-native (sm_100a) Gibbs/FFBS path of joe5saia/Hmc.jl behind the reference's own interface.

The directory name contains a dot, so import it through the root shim:  `import hmc_jl_b200`.
Layout: csrc/ (CUDA kernels + C ABI), lib/ (built libhmcgpu.so), binding.py (ctypes over include/hmcgpu.h),
api.py (mirror of Hmc.estopt / Hmc.estimatemodel / Hmc.estimatesignals!), julia/HmcGPU.jl (the ccall binding a Julia user loads).
"""
from . import build  # noqa: F401
from .api import (EstOpt, estimatemodel, estimatesignals, estimate_windows, shard_windows, expanding_windows,  # noqa: F401
                  gather_window_summaries, saveresults, write_summaries, write_diagnostics, write_predictive, write_ranked,
                  write_onestep, pseudo_residuals, compare_waic, compare_loo, write_loo, predictive_quantiles, forecastinsample,
                  signal_summaries, calcdispersion, calccorr, write_signal_summaries, write_dispersion,
                  makeparams_states, sample_and_forecast_all, saveinsampleforecasts, smoothStates, savesmoothresults)
from .binding import (Context, HmcGpuError, Plan, ProblemSpec, estimate, estimate_multi, load, lib_path,  # noqa: F401
                      FLAG_REF_Q1, FLAG_DRAWS, FLAG_SUMMARY, FLAG_SMOOTHED_MEAN, FLAG_LOGLIK, FLAG_FILTERED_MEAN, FLAG_DIAGNOSTICS,
                      FLAG_PREDICTIVE, FLAG_RANKED, FLAG_ONESTEP, FLAG_LOO, Predictive, Ranked, Onestep, Loo,
                      SYMBOLS)
