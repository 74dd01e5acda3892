"""B200-native guided-proposal path updates behind the DiffusionMCMCTools.jl API.

The directory name carries a dot, so import it through the shim at the repo root:  `import dmt_b200`.
"""
from . import _lib, configs, host, param_names, hetero  # noqa: F401
from .hetero import HeterogeneousBlockEnsemble, HeterogeneousEnsemble  # noqa: F401
from .param_names import ParamNamesAllObs, ParamNamesBlock, ParamNamesRecording, ParamNamesUnit  # noqa: F401
from ._lib import Ctx, DmtError  # noqa: F401
from .host import (BlockEnsemble, SamplingEnsemble, accept_reject_proposal_path, accpt_rate, draw_proposal_path,  # noqa: F401
                   fetch_ll, fetch_ll_o, find_W_for_X, ll_of_accepted, loglikhd, loglikhd_o, recompute_guiding_term, save_ll,
                   set_obs, set_proposal_law, shard_slice, save_state, load_state, blocking_sweep, enable_guiding_cache, swap_ll, swap_paths, swap_PP, swap_WW, swap_XX, set_ll, set_accepted, recompute_path, is_critical_update, PathSaver, PathMoments,
                   set_rho_chains, enable_rho_adaptation, adapt_rho, disable_rho_adaptation)
