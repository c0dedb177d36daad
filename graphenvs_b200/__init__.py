"""graphenvs_b200 -- B200-native batched engine for the GraphEnvs hot path (step / mask / obs).

Public surface:
  make(id, **kwargs)                 gymnasium-shaped single env (reference ids and kwargs)
  make_batched(id, num_envs, ...)    batched vector env with the same per-env semantics
  BatchedGraphEnv                    the engine class behind both (sample_logits: policy-driven action draw;
                                     save_states / load_states / gather_instances / like: branching for search decoders)
  masked_log_prob(logits, mask_bits, actions)   differentiable masked log-prob + entropy for the update (policy.py)
  BeamSearch(venv, width)            beam search / multi-start decoding of a policy on the device (beam.py)
  StochasticBeamSearch(venv, width, seed)   width distinct sequences per instance sampled without replacement (beam.py)
  MCTS(venv, num_simulations, c_puct)   Monte Carlo tree search with PUCT selection on the device (mcts.py)
  utils.vectorize_graph / devectorize_graph / get_env_info   (graph_envs/utils.py layout contract)
"""
from .spec import ENV_SPECS, get_env_info, get_num_features  # noqa: F401

name = "graphenvs_b200"
__version__ = "0.1.0"


def __getattr__(attr):  # lazy: keeps `import graphenvs_b200` cheap and torch-free until needed
    if attr in ("BatchedGraphEnv", "EnvStates", "STATE_DYNAMIC", "STATE_CLOCK", "STATE_STATS", "STATE_ALL"):
        from . import batch
        return getattr(batch, attr)
    if attr in ("make", "make_batched", "register_with_gymnasium", "registry"):
        from . import registration
        return getattr(registration, attr)
    if attr == "masked_log_prob":
        from .policy import masked_log_prob
        return masked_log_prob
    if attr in ("BeamSearch", "StochasticBeamSearch"):
        from . import beam
        return getattr(beam, attr)
    if attr == "MCTS":
        from .mcts import MCTS
        return MCTS
    if attr in ("Instance", "generate_instance"):
        from . import instances
        return getattr(instances, attr)
    raise AttributeError(attr)
