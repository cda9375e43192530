"""dpomp-b200: the particle-filter hot path of DiscretePOMP.jl on B200 (hand-written CUDA for sm_100a behind a C ABI).

The package directory is named after the reference (`discretepomp.jl_b200`), which is not an importable identifier;
import it through the repo-root shim module `dpomp_b200`:

    import dpomp_b200 as dp
    model = dp.generate_model("SIS", [100, 1])
    y = dp.get_observations("tests/golden/pooley.csv")
    f = dp.get_particle_filter_lpdf(model, y, np=200)
    f([0.003, 0.1])

Exported names are those of the reference's public API that lie on the path (src/DiscretePOMP.jl:59-67).
"""
from .structs import (DPOMPModel, Event, HiddenMarkovModel, ImportanceSample, MCMCSample, Observation, Particle,
                      RejectionSample, SimResults)
from .examples import (CountObsModel, GaussianObsModel, UniformProduct, dmy_obs_fn, generate_custom_model, generate_model,
                       generate_trans_fn, generate_weak_prior, partial_binomial_obs_model, partial_gaussian_obs_model,
                       partial_negbin_obs_model, partial_poisson_obs_model)
from .rate_table import ModelCompileError, compile_obs_table, compile_rate_table
from .utils import get_observations
from .particle_filter import (C_DF_ESS_CRIT, C_DF_PF_P, DeviceModel, FilteredStates, ParticleFilter, compile_model,
                              compute_ess, device_model, estimate_likelihood, get_filtered_states, get_log_pdf_fn,
                              get_particle_filter_lpdf, get_private_model)
from .resample import rs_multinomial, rs_stratified, rs_systematic, rsp_indices
from .distributed import Comm, migration_plan, partition_bounds, partition_owner
from .ibis import (compute_is_mu_covar, get_mv_param, get_prop_density, run_ibis_analysis, run_pibis)
from .mcmc import gelman_diagnostic_sre, handle_rej_samples, run_pmcmc, run_pmcmc_analysis
from .mbp_ibis import MbpParticles, run_mbp_ibis
from .mbp_mcmc import generate_x0, run_mbp_mcmc, run_mcmc_analysis
from .da_mcmc import run_std_mcmc
from .sim import generate_observations, gillespie_sim, save_to_file
from .arq import (ARQMCMCSample, ARQModel, GridPoint, GridRequest, LikelihoodModel, adapt_jw, get_grid_points, get_theta_f,
                  run_arq_mcmc_analysis)
from .mcomp import ModelComparisonResults, run_model_comparison, run_model_comparison_analysis
from . import _capi
